// ksg_api.cu — host side of the C-ABI in include/ksg.h: owns the device-resident map (spatial block hash +
// tile pool), the per-frame scratch, and enqueues the kernel family of ksg_kernels.cuh.
// Compiled for sm_100a only, with -fmad=false (bit-exact index arithmetic, see ksg_device.cuh).
#include <cuda_runtime.h>
#include <cub/cub.cuh>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/ksg.h"
#include "ksg_kernels.cuh"
#include "ksg_chain.cuh"
#include "ksg_hot.cuh"
#include "ksg_bundle_order.cuh"
#include "ksg_fast.cuh"
#include "ksg_fast3.cuh"
#include "ksg_voxel.cuh"
#include "ksg_merge.cuh"
#include "ksg_eval.cuh"
#include "ksg_mesh.cuh"

using namespace ksg;

namespace {

thread_local std::string g_last_error;

#define KSG_CUDA(call)                                                                              \
  do {                                                                                              \
    cudaError_t e_ = (call);                                                                        \
    if (e_ != cudaSuccess) {                                                                        \
      char buf_[512];                                                                               \
      snprintf(buf_, sizeof(buf_), "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
      return fail(KSG_ERR_CUDA, buf_);                                                              \
    }                                                                                               \
  } while (0)

inline int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }
inline uint32_t round_up(uint32_t v, uint32_t m) { return (v + m - 1) / m * m; }
inline int grid_for(long long n, int block) { return (int)std::max<long long>(1, (n + block - 1) / block); }

}  // namespace

struct ksg_integrator {
  ksg_config cfg{};
  DevCfg dc{};
  int device = 0;
  int sm_count = 148;
  cudaStream_t own_stream = nullptr;
  std::string err;
  int deferred_status = 0;

  // map
  MapRef map{};
  uint32_t ht_cap = 0;
  Luts h_luts{};
  Luts* d_luts = nullptr;
  Counters* d_cnt = nullptr;
  Counters* h_cnt = nullptr;  // pinned
  int frame_stamp = 0;
  int64_t num_blocks = 0;
  int64_t last_blocks_touched = 0;

  // per-frame scratch
  int cap_points = 0;
  float4 *pt_pC = nullptr, *pt_pG = nullptr;
  uint8_t *pt_label = nullptr, *pt_flags = nullptr;
  uint32_t* pt_color = nullptr;
  uint64_t* pt_key = nullptr;
  uint8_t *flags8 = nullptr, *is_last = nullptr;  // flags8: 2*cap bytes
  int* pix_list = nullptr;
  int* point_of_seq = nullptr;
  uint32_t *sq_keys = nullptr, *sq_keys_out = nullptr;
  uint32_t *iota = nullptr;

  // fast
  int *start_head = nullptr, *start_next = nullptr, *start_min = nullptr, *start_max = nullptr;
  uint32_t* start_val = nullptr;
  uint8_t* start_mixed = nullptr;
  uint8_t *clear_ff = nullptr, *clear_00 = nullptr;
  uint32_t *start_table = nullptr;
  uint64_t set_offset = 0;  // both ApproxHashSets share reset times, hence one offset (fast.cpp:165-170)
  int64_t reset_counter = 0;
  int* cast_seq = nullptr;
  float4* ray_param = nullptr;
  uint8_t *ray_label = nullptr, *ray_flags = nullptr;
  uint32_t* ray_color = nullptr;
  int *nsteps = nullptr, *H = nullptr, *L = nullptr;
  RayState* ray_state = nullptr;
  long long* ext_off = nullptr;
  int* eval_sweep = nullptr;
  int sweep_counter = 0;
  ObsBuf ob{};

  // merged
  uint64_t* ks_sorted = nullptr;
  uint32_t* seq_sorted = nullptr;
  int *bstart = nullptr, *bundle_f = nullptr;
  float *hist = nullptr, *tmp = nullptr, *tmp4 = nullptr;   // tmp4: rows of tmp at a 4-float stride (k_voxel_apply_short_t)
  uint64_t* b_key = nullptr;
  long long* b_base = nullptr;
  // merged, KSG_BUNDLE_ORDER_LIBSTDCXX
  std::vector<std::pair<int, uint32_t>> bord_phases;   // (first insertion index, bucket count) of every rehash phase
  uint32_t* bord_hash = nullptr;
  int* bundle_f2 = nullptr;
  int* bord_scratch = nullptr;       // one allocation behind every array of BordBuf
  unsigned long long* d_scan_tot = nullptr;   // per-CTA totals of k_bundle_scan
  BordBuf bord{};

  // merged, hot_voxel_mode = 1 (ksg_hot.cuh)
  bool hot_enabled = false;
  HotSeg* d_hot_segs = nullptr;
  HotSeg* h_hot_segs = nullptr;      // pinned
  int *d_hot_counts = nullptr;       // [0] segments found, [1] chunks that fell back to the plain loop (accumulated)
  int *d_hot_chunk_seg = nullptr, *h_hot_chunk_seg = nullptr, *d_hot_guess = nullptr;
  double* d_hot_sums = nullptr;
  ChainTable* d_hot_tables = nullptr;
  float* d_hot_prior = nullptr;
  int* d_hot_same = nullptr;          // hot_voxel_mode 2
  long long hot_chunk_cap = 0;
  int64_t hot_segments_total = 0, hot_chunks_total = 0;

  // records
  uint64_t *rec_a = nullptr, *rec_b = nullptr;
  long long rec_cap = 0;
  long long* tile_begin = nullptr;
  long long tile_cap = 0;
  void* cub_temp = nullptr;
  size_t cub_temp_bytes = 0;

  // host staging (pinned) + device input buffers for the host-buffer entry points
  uint8_t* h_stage = nullptr;
  size_t h_stage_bytes = 0;
  uint8_t* d_in = nullptr;
  size_t d_in_bytes = 0;

  // export staging
  uint8_t* d_exp = nullptr;
  size_t d_exp_bytes = 0;
  int* d_exp_slots = nullptr;
  int exp_slots_cap = 0;

  // fast, round-2 frame driver (ksg_fast.cuh): no host read-back inside the frame
  bool fast_v2 = false;
  FastCounters* d_fc = nullptr;
  FastCounters* h_fc = nullptr;      // pinned
  long long* d_prof = nullptr;       // [kProfSlots] solver counters of the last profiled frame (allocated when profiling is first enabled)
  int *blk_cnt = nullptr, *blk_off = nullptr, *warp_cnt = nullptr, *warp_off = nullptr, *seq_of_i = nullptr;
  uint32_t* keys32 = nullptr;
  int *tile_cnt = nullptr, *tile_slot = nullptr;
  TileDesc* tile_list = nullptr;
  int solve_grid = 0, apply_fast_smem = 0;
  int solver = 3;                    // 3: rank-group solver (ksg_fast3.cuh), 2: first persistent formulation (k_fast_solve)
  int solve_threads = kSolveThreads; // tuning knobs (environment): KSG_SOLVE_THREADS, KSG_SOLVE_CTAS_PER_SM, KSG_GROUP0, KSG_GROUP_MUL
  int group0 = kGroup0, group_mul = 4;
  Cand* cand16 = nullptr;
  OvfEnt* ovf = nullptr;
  RayRec* rayrec = nullptr;
  int ovf_cap = 0;
  int *mixed_list = nullptr, *m_list = nullptr, *blk_run = nullptr;
  // update log (ksg_set_update_log): one entry per voxel the last frame updated
  VoxelUpdate *d_log_head = nullptr, *h_log_head = nullptr;
  float *d_log_prior = nullptr, *h_log_prior = nullptr;
  int log_cap = 0;
  uint64_t* stamp64 = nullptr;       // [2][2^20] toggle stamps of solver 3
  int solve_smem = 0;
  double clock_khz = 1965000.0;
  // frames whose counters have not been read back yet (at most two: the counter copies land in two pinned slots)
  Counters* h_cnt_base = nullptr;    // [2] pinned; h_cnt points at the slot read last
  FastCounters* h_fc_base = nullptr; // [2] pinned
  cudaEvent_t ev_frame_s[2] = {nullptr, nullptr};   // recorded behind the frame's counter copy
  int pend[2] = {0, 0};
  int n_pend = 0, next_slot = 0;
  // pipelined host-buffer entry (ksg_integrate_depth_async): the H2D copy of frame t+1 overlaps the kernels of frame t
  cudaStream_t copy_stream = nullptr;
  uint8_t* d_in2[2] = {nullptr, nullptr};
  uint8_t* h_stage2[2] = {nullptr, nullptr};
  size_t in2_bytes[2] = {0, 0};
  cudaEvent_t ev_copy[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
  bool in2_used[2] = {false, false};
  int in_slot = 0;
  ksg_frame_stats stash[4];
  int n_stash = 0;
  int pending_iterations = 0;
  long long pending_records = -1;    // legacy paths know the record count on the host; -1: read it from the counters

  // merged, round-2 per-voxel apply (ksg_voxel.cuh)
  bool voxel_apply = false;
  VoxelQueues vq{};
  cudaStream_t aux_stream = nullptr, aux_stream2 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join2 = nullptr;
  // both measured SLOWER than what they were meant to replace (profiles/r02/bench_full_9.json vs bench_merged2_nohotk.json: the hot
  // voxels' critical path is the TSDF weight recurrence, which a producer / consumer ring does not shorten; the warp-wide ray walk costs
  // more in rank searches than the scattered stores it saves) - kept as opt-in experiments: KSG_HOT_KERNEL=1, KSG_EMIT_WARP=1
  bool hot_kernel = false;
  bool emit_warp = false;
  // shape of the two per-voxel kernels (environment: KSG_LONG_THREADS, KSG_LONG_GRID, KSG_SHORT_CTAS): the short-segment kernel is
  // capped at short_ctas CTAs per SM through a dynamic shared-memory reservation so that a CTA of the long-segment kernel (128
  // registers per thread) always finds room beside it - otherwise the two kernels run back to back
  // (measured on merged2, profiles/r02/tuning_10.log: 6 CTAs/SM -> 148 fps, 4 + long 128 x 296 -> 163, 3 -> 166)
  int long_threads = 256, long_grid = 0, short_ctas = 3, short_smem = 0;
  bool short_thread = false;         // merged, C <= 32: k_voxel_apply_short_t
  // the non-hot long segments (0.3 ms standalone) run behind the short kernel on its stream instead of beside it (KSG_LONG_SERIAL=0:
  // beside it): 202 against 199 frames/s with two short-kernel CTAs per SM (profiles/r02/tuning_18.log)
  bool long_serial = true;
  int deep_threads = 128;            // block size of the hot-voxel instance (KSG_DEEP_THREADS): one warp per chain, 148 x 4 warps
  bool deep_hot = true;              // merged, C <= 32: the hot voxels go to the deep-pipeline instance of k_voxel_apply_long (KSG_DEEP_HOT=0: off)
  // its CTAs per SM (KSG_SHORT_T_CTAS).  The frame is bound by the long-segment kernel (1184 warps, 128 registers each); whatever the
  // short kernel takes from it costs more than it gains: merged2 1 -> 178 fps, 2 -> 166, 3 -> 166, 4 -> 170, warp-per-voxel kernel 170
  // (profiles/r02/tuning_12.log)
  int short_t_ctas = 2;              // (1 while the hot chains ran inside the long-segment kernel: tuning_12.log; 2 with the deep instance: tuning_18.log)
  int hot_smem = 0;

  long long* tile_debug = nullptr;  // optional per-tile (records, cycles) trace
  int sweeps_per_sync = 1;
  int first_batch = 4;
  bool persistent_eval = true;
  unsigned int* d_gridbar = nullptr;
  int eval_grid = 0;   // sweeps launched before the first read-back (a 640x480 frame needs 6-8)
  int apply_smem = 0;
  int apply_nch = 1;
  bool use_tma = true;

  // profiling
  bool profiling = false;
  cudaEvent_t ev[KSG_NUM_PHASES + 1] = {};
  double phase_ms[KSG_NUM_PHASES] = {};
  int64_t prof_frames = 0;
  int64_t n_launches = 0, n_libcalls = 0;

  int fail(int code, const char* msg) { err = msg; g_last_error = msg; return code; }
};

namespace {

int validate(const ksg_config* c, std::string& why) {
  if (!c) { why = "null config"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->abi_version != KSG_ABI_VERSION) { why = "abi_version mismatch"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->integrator_type != KSG_INTEGRATOR_FAST && c->integrator_type != KSG_INTEGRATOR_MERGED) {
    why = "Unknown Semantic/TSDF integrator type (factory.cpp:83)"; return KSG_ERR_INVALID_ARGUMENT; }
  const int v = c->voxels_per_side;
  if (v <= 0 || (v & (v - 1)) || v > 64) { why = "voxels_per_side must be a power of two <= 64"; return KSG_ERR_INVALID_ARGUMENT; }
  if (!(c->voxel_size > 0.0f)) { why = "voxel_size must be positive"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->num_labels < 2 || c->num_labels > 256) { why = "num_labels must be in [2, 256]"; return KSG_ERR_INVALID_ARGUMENT; }
  const float p = c->semantic_measurement_probability;  // base.cpp:98-107
  if (!(p > 0.0f && p < 1.0f) || !((1.0f - p) > 0.0f) || !(std::log(p) > std::log(1.0f - p))) {
    why = "semantic_measurement_probability must satisfy 0 < 1-p < p < 1 (base.cpp:98-107)"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->integration_order_mode != KSG_ORDER_MIXED && c->integration_order_mode != KSG_ORDER_SORTED) {
    why = "unknown integration_order_mode"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->color_mode < 0 || c->color_mode > 2) { why = "Unknown semantic color mode (base.cpp:186-190)"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->max_points <= 0 || c->max_points > (1 << kRecOrdBits)) { why = "max_points must be in (0, 2^23]"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->max_blocks <= 0) { why = "max_blocks must be positive"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->shard_count < 0 || (c->shard_count > 1 && (c->shard_rank < 0 || c->shard_rank >= c->shard_count))) {
    why = "shard_rank must be in [0, shard_count)"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->max_consecutive_ray_collisions < 0) { why = "max_consecutive_ray_collisions < 0"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->merged_bundle_order != KSG_BUNDLE_ORDER_CANONICAL && c->merged_bundle_order != KSG_BUNDLE_ORDER_LIBSTDCXX) {
    why = "unknown merged_bundle_order"; return KSG_ERR_INVALID_ARGUMENT; }
  if (c->hot_voxel_mode < 0 || c->hot_voxel_mode > 2) { why = "unknown hot_voxel_mode"; return KSG_ERR_INVALID_ARGUMENT; }
  return KSG_OK;
}

template <typename Tp>
cudaError_t dmalloc(Tp** p, size_t count) { return cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(Tp)); }

void free_all(ksg_integrator* h) {
  cudaSetDevice(h->device);
  void* ptrs[] = {h->map.ht_keys, h->map.ht_slot, h->map.new_list, h->map.pool, h->map.slot_key, h->map.touched_stamp,
                  h->map.touched_list, h->d_luts, h->d_cnt, h->pt_pC, h->pt_pG, h->pt_label, h->pt_flags, h->pt_color, h->pt_key,
                  h->flags8, h->is_last, h->pix_list, h->point_of_seq, h->sq_keys, h->sq_keys_out, h->iota,
                  h->start_next, h->start_min, h->clear_ff, h->clear_00, h->start_table, h->cast_seq, h->ray_param, h->ray_label, h->ray_flags,
                  h->ray_color, h->nsteps, h->H, h->L, h->ray_state, h->ext_off, h->eval_sweep, h->ob.slot_stamp, h->ob.cand_pos, h->ob.bkt, h->ob.cand_val, h->ob.cand_order,
                  h->ob.cand_next, h->ob.table, h->ks_sorted, h->seq_sorted, h->bstart, h->bundle_f, h->hist,
                  h->tmp, h->tmp4, h->b_key, h->b_base, h->bord_hash, h->bord_scratch, h->d_scan_tot, h->bundle_f2, h->d_hot_segs, h->d_hot_counts, h->d_hot_chunk_seg, h->d_hot_guess, h->d_hot_sums,
                  h->d_hot_tables, h->d_hot_prior, h->d_hot_same, h->tile_debug, h->d_gridbar, h->d_fc, h->d_prof, h->blk_cnt, h->blk_off, h->warp_cnt, h->warp_off, h->seq_of_i, h->keys32,
                  h->tile_cnt, h->tile_slot, h->tile_list, h->cand16, h->ovf, h->rayrec, h->mixed_list, h->m_list, h->blk_run, h->stamp64, h->d_log_head, h->d_log_prior, h->vq.long_items, h->vq.counters, h->rec_a, h->rec_b, h->tile_begin, h->cub_temp, h->d_in, h->d_exp, h->d_exp_slots};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (h->h_cnt_base) cudaFreeHost(h->h_cnt_base);
  if (h->h_log_head) cudaFreeHost(h->h_log_head);
  if (h->h_log_prior) cudaFreeHost(h->h_log_prior);
  if (h->h_fc_base) cudaFreeHost(h->h_fc_base);
  for (int i = 0; i < 2; ++i) {
    if (h->ev_frame_s[i]) cudaEventDestroy(h->ev_frame_s[i]);
    if (h->ev_copy[i]) cudaEventDestroy(h->ev_copy[i]);
    if (h->ev_free[i]) cudaEventDestroy(h->ev_free[i]);
    if (h->d_in2[i]) cudaFree(h->d_in2[i]);
    if (h->h_stage2[i]) cudaFreeHost(h->h_stage2[i]);
  }
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev_join2) cudaEventDestroy(h->ev_join2);
  if (h->aux_stream2) cudaStreamDestroy(h->aux_stream2);
  if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
  if (h->h_stage) cudaFreeHost(h->h_stage);
  if (h->h_hot_segs) cudaFreeHost(h->h_hot_segs);
  if (h->h_hot_chunk_seg) cudaFreeHost(h->h_hot_chunk_seg);
  for (auto& e : h->ev) if (e) cudaEventDestroy(e);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
}

__global__ void k_iota(uint32_t* p, int n) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = (uint32_t)i; }

// "sorted" integration order (voxblox SortedThreadSafeIndex, A.3): key = squared norm of the point
__global__ void k_sqnorm(FrameIn in, const Counters* cnt, int capacity, uint32_t* keys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= capacity) return;
  if (i >= cnt->n_points) { keys[i] = 0xFFFFFFFFu; return; }
  F3 pC;
  if (in.depth) {
    const int pix = in.pix_list[i];
    const int v = pix / in.width, u = pix - v * in.width;
    const float d = in.depth[pix];
    pC = f3(((float)u - in.cx) * d * in.constant_x, ((float)v - in.cy) * d * in.constant_y, d * in.z_scale);
  } else pC = f3(in.xyz[3 * i], in.xyz[3 * i + 1], in.xyz[3 * i + 2]);
  keys[i] = __float_as_uint(dot3(pC, pC));
}

int reset_map(ksg_integrator* h, cudaStream_t s) {
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaMemsetAsync(h->map.ht_keys, 0xFF, sizeof(uint64_t) * h->ht_cap, s));
  KSG_CUDA(cudaMemsetAsync(h->map.ht_slot, 0xFF, sizeof(int) * h->ht_cap, s));
  KSG_CUDA(cudaMemsetAsync(h->map.touched_stamp, 0, sizeof(int) * h->ht_cap, s));
  KSG_CUDA(cudaMemsetAsync(h->d_cnt, 0, sizeof(Counters), s));
  if (h->start_table) KSG_CUDA(cudaMemsetAsync(h->start_table, 0xFF, sizeof(uint32_t) * kSetSize, s));
  if (h->ob.table) KSG_CUDA(cudaMemsetAsync(h->ob.table, 0xFF, sizeof(uint32_t) * kSetSize, s));
  if (h->ob.slot_stamp) KSG_CUDA(cudaMemsetAsync(h->ob.slot_stamp, 0, sizeof(int) * kSetSize, s));
  if (h->d_fc) KSG_CUDA(cudaMemsetAsync(h->d_fc, 0, sizeof(FastCounters), s));
  if (h->stamp64) {   // (sweep 0, nobody): max word 0, min word all ones
    KSG_CUDA(cudaMemsetAsync(h->stamp64, 0x00, sizeof(uint64_t) * kSetSize, s));
    KSG_CUDA(cudaMemsetAsync(h->stamp64 + kSetSize, 0xFF, sizeof(uint64_t) * kSetSize, s));
  }
  if (h->tile_cnt) KSG_CUDA(cudaMemsetAsync(h->tile_cnt, 0, sizeof(int) * (size_t)h->ht_cap * h->dc.tiles_per_block, s));
  h->n_pend = 0; h->n_stash = 0;
  std::memset(h->h_cnt_base, 0, 2 * sizeof(Counters));
  h->sweep_counter = 0;
  h->set_offset = 0;
  h->reset_counter = 0;
  h->num_blocks = 0;
  h->frame_stamp = 0;
  h->last_blocks_touched = 0;
  h->deferred_status = 0;
  KSG_CUDA(cudaStreamSynchronize(s));
  return KSG_OK;
}

struct InputDesc {
  const float* d_xyz = nullptr;
  const uint8_t* d_rgba = nullptr;
  const uint8_t* d_labels = nullptr;
  const float* d_depth = nullptr;
  const uint8_t* d_label_img = nullptr;
  int width = 0, height = 0;
  double K[4] = {0, 0, 0, 0};   // fx fy cx cy as the reference holds them (sensor_msgs/CameraInfo: float64)
  double unit_scaling = 1.0;    // DepthTraits<T>::toMeters(T(1)) as double: 1 (float32 metres) or double(0.001f) (uint16 millimetres)
  float z_scale = 1.0f;
  const uint32_t* d_color_img = nullptr;
  int64_t n = 0;  // points (points entry) or pixels (depth entry)
  int freespace = 0;
};

int fetch_counters(ksg_integrator* h, cudaStream_t s) {
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaMemcpyAsync(h->h_cnt, h->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, s));
  KSG_CUDA(cudaStreamSynchronize(s));
  return KSG_OK;
}

const char* err_text(int e) {
  switch (e) {
    case 1: return "invalid argument: a semantic label >= num_labels (CHECK_LT fast.cpp:134 / merged.cpp:278)";
    case 2: return "observed-set solver did not converge within its sweep budget";
    case 3: return "block pool / hash table full: raise ksg_config.max_blocks";
    case 4: return "per-frame scratch full: raise ksg_config.max_ray_steps / max_updates";
    case 5: return "voxel or block index outside the supported range";
    default: return "device-side error";
  }
}

// hot_voxel_mode = 1: finish the log-probability rows of the frame's hot voxels ahead of the tile kernel (ksg_hot.cuh).
// Returns the number of hot segments (0: nothing to do) through *n_hot.
int hot_voxel_prepass(ksg_integrator* h, cudaStream_t s, const Xform& T, const float4* bundle_param, long long n_records, int* n_hot) {
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  const DevCfg& dc = h->dc;
  *n_hot = 0;
  KSG_CUDA(cudaMemsetAsync(h->d_hot_counts, 0, sizeof(int), s));
  ++h->n_launches;
  k_hot_find<<<grid_for(n_records, 256), 256, 0, s>>>(dc, h->map, h->rec_b, n_records, h->d_hot_segs, h->d_hot_counts);
  int found = 0;
  KSG_CUDA(cudaMemcpyAsync(&found, h->d_hot_counts, sizeof(int), cudaMemcpyDeviceToHost, s));
  KSG_CUDA(cudaStreamSynchronize(s));
  const int n = std::min(found, kHotMaxSegs);
  if (n <= 0) return KSG_OK;
  KSG_CUDA(cudaMemcpyAsync(h->h_hot_segs, h->d_hot_segs, sizeof(HotSeg) * (size_t)n, cudaMemcpyDeviceToHost, s));
  KSG_CUDA(cudaStreamSynchronize(s));
  std::sort(h->h_hot_segs, h->h_hot_segs + n, [](const HotSeg& a, const HotSeg& b) { return a.begin < b.begin; });
  long long chunks = 0;
  int kept = 0;
  for (int i = 0; i < n; ++i) {                       // segments that do not fit the chunk scratch stay on the ordinary path
    HotSeg& g = h->h_hot_segs[i];
    if (chunks + g.n_chunks > h->hot_chunk_cap) break;
    g.first_chunk = (int)chunks;
    for (int k = 0; k < g.n_chunks; ++k) h->h_hot_chunk_seg[chunks + k] = i;
    chunks += g.n_chunks;
    ++kept;
  }
  if (kept == 0) return KSG_OK;
  KSG_CUDA(cudaMemcpyAsync(h->d_hot_segs, h->h_hot_segs, sizeof(HotSeg) * (size_t)kept, cudaMemcpyHostToDevice, s));
  KSG_CUDA(cudaMemcpyAsync(h->d_hot_chunk_seg, h->h_hot_chunk_seg, sizeof(int) * (size_t)chunks, cudaMemcpyHostToDevice, s));
  const int nch = (int)chunks;
  h->n_launches += 4;
  k_hot_chunk_sums<<<grid_for((long long)nch * 32, 128), 128, 0, s>>>(dc.C, h->d_hot_segs, h->d_hot_chunk_seg, nch, h->rec_b, h->tmp, h->d_hot_sums);
  k_hot_guess<<<grid_for((long long)kept * 32, 128), 128, 0, s>>>(dc.C, h->d_hot_segs, kept, h->map.pool, h->d_hot_sums, h->d_hot_guess);
  k_hot_chunk_tables<<<nch, 128, sizeof(float) * (size_t)dc.C * kHotColStride, s>>>(dc.C, h->d_hot_segs, h->d_hot_chunk_seg, h->rec_b, h->tmp,
                                                                                  h->d_hot_guess, h->d_hot_tables);
  k_hot_apply<<<grid_for((long long)kept * 32, 128), 128, 0, s>>>(dc.C, h->d_hot_segs, kept, h->map.pool, h->rec_b, h->tmp, h->d_hot_guess,
                                                                  h->d_hot_tables, h->d_hot_prior, h->d_hot_counts + 1);
  if (h->cfg.hot_voxel_mode == 2) {
    KSG_CUDA(cudaMemsetAsync(h->d_hot_same, 0x01, sizeof(int) * (size_t)kept, s));   // 0x01010101: non-zero = "same" until refuted
    ++h->n_launches;
    k_hot_tsdf_same<<<nch, 128, 0, s>>>(dc, T, h->d_hot_segs, h->d_hot_chunk_seg, h->map.pool, h->rec_b, bundle_param, h->d_hot_same);
  }
  KSG_CUDA(cudaGetLastError());
  h->hot_segments_total += kept;
  h->hot_chunks_total += chunks;
  *n_hot = kept;
  return KSG_OK;
}


void fill_stats(ksg_integrator* h, ksg_frame_stats* stats) {
  std::memset(stats, 0, sizeof(*stats));
  stats->points_in = h->h_cnt->n_points;
  stats->points_valid = h->h_cnt->n_valid;
  stats->rays_cast = h->h_cnt->n_cast;
  stats->ray_steps = (int64_t)h->h_cnt->ray_steps;
  stats->voxel_updates = (int64_t)h->h_cnt->n_records - (int64_t)h->h_cnt->n_skipped;
  stats->blocks_allocated = h->num_blocks;
  stats->blocks_touched = h->h_cnt->n_blocks_touched;
  stats->tiles_touched = h->h_cnt->n_tiles;
  stats->fixpoint_iterations = h->h_fc ? h->h_fc->sweeps_last : 0;
}

// Completes the OLDEST frame whose counters are still in flight (fast, round-2 driver): waits for its counter copy, mirrors the
// counters on the host and reports a device-side error.
int finish_oldest(ksg_integrator* h, ksg_frame_stats* stats) {
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  if (h->n_pend <= 0) return KSG_OK;
  const int slot = h->pend[0];
  h->pend[0] = h->pend[1];
  --h->n_pend;
  KSG_CUDA(cudaEventSynchronize(h->ev_frame_s[slot]));
  h->h_cnt = h->h_cnt_base + slot;
  if (h->h_fc_base) h->h_fc = h->h_fc_base + slot;
  h->num_blocks = h->h_cnt->pool_count;
  h->last_blocks_touched = h->h_cnt->n_blocks_touched;
  if (h->profiling && h->h_fc) {
    // events: 0 frame start, 1 before the solve kernel, 2 after it, 3 after the tile kernel; the solve kernel's own phases come from
    // the clock64 marks block 0 left in FastCounters::timeline
    float a = 0, b = 0, c = 0, tot = 0;
    cudaEventElapsedTime(&a, h->ev[0], h->ev[1]); cudaEventElapsedTime(&b, h->ev[1], h->ev[2]);
    cudaEventElapsedTime(&c, h->ev[2], h->ev[3]); cudaEventElapsedTime(&tot, h->ev[0], h->ev[3]);
    const long long* tl = h->h_fc->timeline;
    const int sweeps_end = (int)tl[kTimelineSlots - 1];
    const int tb = kTimelineSlots - 12;
    const double span = (double)(tl[tb + 4] - tl[0]);
    if (span > 0 && sweeps_end >= 3 && sweeps_end <= tb) {
      const double k = (double)b / span;
      h->phase_ms[0] += a + k * (double)(tl[2] - tl[0]);                 // count + classify + start set + compaction + ray set-up
      h->phase_ms[1] += k * (double)(tl[tb] - tl[2]);                    // observed-set sweeps
      h->phase_ms[2] += k * (double)(tl[tb + 1] - tl[tb]);               // table commit + ray emit / block allocation
      h->phase_ms[3] += k * (double)(tl[tb + 4] - tl[tb + 1]);           // records -> tile segments (count, allocate + new blocks, scatter)
    } else { h->phase_ms[0] += a; h->phase_ms[1] += b; }
    h->phase_ms[5] += c;
    h->phase_ms[6] += tot;
    h->prof_frames += 1;
  }
  if (stats) fill_stats(h, stats);
  const int dev_err = h->h_cnt->err;
  if (dev_err) {
    h->deferred_status = dev_err;  // the map may be inconsistent from here on
    return fail(dev_err, err_text(dev_err));
  }
  return KSG_OK;
}
// Completes every outstanding frame; `stats` receives the newest frame's counters.
int finish_frame(ksg_integrator* h, ksg_frame_stats* stats) {
  while (h->n_pend > 1) { const int rc = finish_oldest(h, nullptr); if (rc) return rc; }
  if (h->n_pend == 1) return finish_oldest(h, stats);
  if (stats) fill_stats(h, stats);
  if (h->deferred_status) return h->fail(h->deferred_status, err_text(h->deferred_status));
  return KSG_OK;
}

// `fast`, round-2 frame driver: five launches, no host read-back inside the frame (ksg_fast.cuh).
int integrate_fast_v2(ksg_integrator* h, const InputDesc& in, const FrameIn& fin, const Xform& T, int cap, cudaStream_t s,
                      ksg_frame_stats* stats) {
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  const bool sorted = h->cfg.integration_order_mode == KSG_ORDER_SORTED;
  // ApproxHashSet resets (fast.cpp:165-170, A.4)
  if ((++h->reset_counter) >= h->cfg.clear_checks_every_n_frames) {
    h->reset_counter = 0;
    if (++h->set_offset >= 10000) {
      h->set_offset = 0;
      KSG_CUDA(cudaMemsetAsync(h->start_table, 0xFF, sizeof(uint32_t) * kSetSize, s));
      KSG_CUDA(cudaMemsetAsync(h->ob.table, 0xFF, sizeof(uint32_t) * kSetSize, s));
    }
  }
  FastFrame f{};
  f.cfg = h->dc; f.T = T; f.in = fin; f.in.pix_list = nullptr; f.in.point_of_seq = nullptr;
  f.luts = h->d_luts; f.cnt = h->d_cnt; f.fc = h->d_fc; f.map = h->map; f.ob = h->ob;
  f.sb = StartBuf{h->start_head, h->start_next, h->start_min, h->start_max, h->start_val, h->start_mixed, h->start_table};
  f.set_offset = h->set_offset;
  f.capacity = cap;
  f.n_count_blocks = (cap + kCountBlock - 1) / kCountBlock;
  f.vec_ok = in.d_depth ? (((uintptr_t)in.d_depth % 16 == 0 && (uintptr_t)in.d_label_img % 4 == 0) ? 1 : 0) : 0;
  f.frame_stamp = h->frame_stamp;
  f.profile = h->profiling ? 1 : 0;
  f.prof = h->d_prof;
  f.seq_of_i = sorted ? h->seq_of_i : nullptr;
  f.block_cnt = h->blk_cnt; f.block_off = h->blk_off; f.warp_cnt = h->warp_cnt; f.warp_off = h->warp_off;
  f.pt_pG = h->pt_pG; f.pt_label = h->pt_label; f.pt_flags = h->pt_flags; f.pt_color = h->pt_color; f.pt_key = h->pt_key;
  f.cast_flag = h->flags8;
  f.cast_seq = h->cast_seq; f.ray_param = h->ray_param; f.ray_label = h->ray_label; f.ray_flags = h->ray_flags; f.ray_color = h->ray_color;
  f.nsteps = h->nsteps; f.H = h->H; f.L = h->L; f.ray_state = h->ray_state; f.ext_off = h->ext_off; f.eval_sweep = h->eval_sweep;
  f.rec = h->rec_a; f.rec_cap = h->rec_cap; f.keys = h->keys32;
  f.tile_cnt = h->tile_cnt; f.tile_slot = h->tile_slot; f.tile_list = h->tile_list; f.tile_cap = h->tile_cap;
  f.o3.cand = h->cand16; f.o3.ext_base = h->ob.ext_base; f.o3.cand_cap = h->ob.cand_cap; f.o3.slot_cnt = h->ob.slot_cnt; f.o3.bkt = h->ob.bkt;
  f.o3.head = h->ob.head; f.o3.ovf = h->ovf; f.o3.ovf_cap = h->ovf_cap; f.o3.stamp_max = h->stamp64; f.o3.stamp_min = h->stamp64 + kSetSize; f.o3.table = h->ob.table;
  f.rayrec = h->rayrec; f.blk_run = h->blk_run;
  f.log_head = h->d_log_head; f.log_prior = h->d_log_prior; f.log_cap = h->log_cap;
  f.group0 = h->group0; f.group_mul = h->group_mul;
  f.s_base = h->start_head; f.s_hmin = h->start_val; f.s_hmax = (uint32_t*)(h->clear_00 + (size_t)kSetSize * 5);
  f.s_visits = (int*)(h->clear_00 + (size_t)kSetSize * 9); f.mixed_list = h->mixed_list; f.m_list = h->m_list;
  const bool s3 = h->solver == 3;

  if (h->profiling) {
    cudaEventRecord(h->ev[0], s);
    KSG_CUDA(cudaMemsetAsync(h->d_fc->dbg, 0, sizeof(h->d_fc->dbg), s));
    KSG_CUDA(cudaMemsetAsync(h->d_prof, 0, sizeof(long long) * kProfSlots, s));
  }
  KSG_CUDA(cudaMemsetAsync(h->clear_ff, 0xFF, (size_t)kSetSize * 16, s));
  KSG_CUDA(cudaMemsetAsync(h->clear_00, 0x00, (size_t)kSetSize * (s3 ? 13 : 5), s));
  KSG_CUDA(cudaMemsetAsync(h->start_min, 0x7F, sizeof(int) * kSetSize, s));
  const int B = 256;
  ++h->n_launches;
  if (in.d_depth) k_fast_count<<<f.n_count_blocks, 256, 0, s>>>(f);
  else k_fast_reset<<<1, 1, 0, s>>>(f);
  if (sorted) {   // voxblox SortedThreadSafeIndex (A.3): stable order by squared norm
    h->n_launches += 3;
    if (in.d_depth) k_fast_sqnorm<<<f.n_count_blocks, 256, 0, s>>>(f, h->sq_keys);
    else k_fast_sqnorm_points<<<grid_for(cap, B), B, 0, s>>>(f, h->sq_keys);
    k_fast_pad_keys<<<grid_for(cap, B), B, 0, s>>>(h->d_cnt, cap, h->sq_keys);
    size_t tb = h->cub_temp_bytes;
    ++h->n_libcalls;
    KSG_CUDA(cub::DeviceRadixSort::SortPairs(h->cub_temp, tb, h->sq_keys, h->sq_keys_out, h->iota, (uint32_t*)h->point_of_seq, cap, 0, 32, s));
    k_fast_invert_perm<<<grid_for(cap, B), B, 0, s>>>(h->d_cnt, (const uint32_t*)h->point_of_seq, h->seq_of_i);
  }
  ++h->n_launches;
  if (in.d_depth) { if (s3) k_fast_classify<true, true><<<f.n_count_blocks, 256, 0, s>>>(f); else k_fast_classify<true, false><<<f.n_count_blocks, 256, 0, s>>>(f); }
  else { if (s3) k_fast_classify<false, true><<<grid_for(cap, B), B, 0, s>>>(f); else k_fast_classify<false, false><<<grid_for(cap, B), B, 0, s>>>(f); }
  const int n_eval_blocks = (cap + kEvalBlock - 1) / kEvalBlock;
  ++h->n_launches;
  if (s3) k_fast_start_eval3<<<n_eval_blocks, kEvalBlock, 0, s>>>(f);
  else k_fast_start_eval<<<n_eval_blocks, kEvalBlock, 0, s>>>(f, n_eval_blocks);
  if (h->profiling) cudaEventRecord(h->ev[1], s);
  {
    int max_sweeps = 4096;   // theory: <= rays + 1 sweeps, practice 6-8; the kernel flags an error rather than spin for ever
    void* args[] = {(void*)&f, (void*)&max_sweeps};
    ++h->n_launches;
    KSG_CUDA(cudaLaunchCooperativeKernel(s3 ? (const void*)k_fast_solve3 : (const void*)k_fast_solve, dim3(h->solve_grid),
                                         dim3(s3 ? h->solve_threads : kSolveThreads), args, s3 ? (size_t)h->solve_smem : 0, s));
  }
  if (h->profiling) cudaEventRecord(h->ev[2], s);
  {
    ApplySrc src{};
    src.param = h->ray_param; src.label = h->ray_label; src.color = h->ray_color; src.tmp = nullptr;
    const int ctas_per_sm = std::max(1, std::min(8, (int)(220 * 1024 / std::max(1, h->apply_fast_smem + 1024))));
    const int grid = h->sm_count * ctas_per_sm;
    ++h->n_launches;
#define KSG_LAUNCH_FAST(TMA, NCH) k_tile_apply_fast<TMA, NCH><<<grid, 512, h->apply_fast_smem, s>>>(f, src)
    if (h->use_tma) {
      switch (h->apply_nch) { case 1: KSG_LAUNCH_FAST(true, 1); break; case 2: KSG_LAUNCH_FAST(true, 2); break;
                              case 4: KSG_LAUNCH_FAST(true, 4); break; default: KSG_LAUNCH_FAST(true, 8); break; }
    } else {
      switch (h->apply_nch) { case 1: KSG_LAUNCH_FAST(false, 1); break; case 2: KSG_LAUNCH_FAST(false, 2); break;
                              case 4: KSG_LAUNCH_FAST(false, 4); break; default: KSG_LAUNCH_FAST(false, 8); break; }
    }
#undef KSG_LAUNCH_FAST
  }
  if (h->profiling) cudaEventRecord(h->ev[3], s);
  KSG_CUDA(cudaGetLastError());
  if (h->n_pend == 2) {   // both counter slots in flight: complete the older frame first (its statistics stay retrievable)
    ksg_frame_stats old_stats;
    const int rco = finish_oldest(h, &old_stats);
    if (h->n_stash < 4) h->stash[h->n_stash++] = old_stats;
    if (rco) return rco;
  }
  const int slot = h->next_slot;
  KSG_CUDA(cudaMemcpyAsync(h->h_cnt_base + slot, h->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, s));
  KSG_CUDA(cudaMemcpyAsync(h->h_fc_base + slot, h->d_fc, sizeof(FastCounters), cudaMemcpyDeviceToHost, s));
  KSG_CUDA(cudaEventRecord(h->ev_frame_s[slot], s));
  h->pend[h->n_pend++] = slot;
  h->next_slot ^= 1;
  if (stats || h->profiling) return finish_frame(h, stats);
  return KSG_OK;
}

int integrate(ksg_integrator* h, const InputDesc& in, const float* T_host, cudaStream_t s, ksg_frame_stats* stats) {
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  if (h->deferred_status) return h->fail(h->deferred_status, err_text(h->deferred_status));
  if (in.n > h->cap_points) return fail(KSG_ERR_INVALID_ARGUMENT, "cloud / frame larger than ksg_config.max_points");
  if (in.n == 0 && h->n_pend > 0) { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  KSG_CUDA(cudaSetDevice(h->device));
  const DevCfg& dc = h->dc;
  const bool fast = h->cfg.integrator_type == KSG_INTEGRATOR_FAST;
  const int cap = (int)in.n;  // host upper bound of the point count
  const int B = 256;
  Xform T{T_host[0], T_host[1], T_host[2], T_host[3], T_host[4], T_host[5], T_host[6]};
  h->frame_stamp += 1;

  if (cap == 0) {
    if (stats) { std::memset(stats, 0, sizeof(*stats)); stats->blocks_allocated = h->num_blocks; }
    if (fast) {  // the sets are still reset (fast.cpp:165-170 runs before any point is looked at)
      if ((++h->reset_counter) >= h->cfg.clear_checks_every_n_frames) {
        h->reset_counter = 0;
        if (++h->set_offset >= 10000) {
          h->set_offset = 0;
          KSG_CUDA(cudaMemsetAsync(h->start_table, 0xFF, sizeof(uint32_t) * kSetSize, s));
          KSG_CUDA(cudaMemsetAsync(h->ob.table, 0xFF, sizeof(uint32_t) * kSetSize, s));
        }
      }
    }
    h->last_blocks_touched = 0;
    return KSG_OK;
  }

  FrameIn fin{};
  fin.xyz = in.d_xyz; fin.rgba = in.d_rgba; fin.labels = in.d_labels;
  fin.depth = in.d_depth; fin.label_img = in.d_label_img; fin.pix_list = h->pix_list;
  fin.point_of_seq = nullptr;
  fin.width = in.width;
  fin.cx = (float)in.K[2]; fin.cy = (float)in.K[3];   // depth_map_to_pointcloud.h:222-223 float center = model_.cx()
  if (in.d_depth) {  // depth_map_to_pointcloud.h:228-230: float constant = unit_scaling / f  (double division)
    fin.constant_x = (float)(in.unit_scaling / in.K[0]);
    fin.constant_y = (float)(in.unit_scaling / in.K[1]);
  }
  fin.z_scale = in.z_scale;
  fin.color_img = in.d_color_img;
  fin.freespace = in.freespace;
  if (fast && h->fast_v2) return integrate_fast_v2(h, in, fin, T, cap, s, stats);

  if (h->profiling) cudaEventRecord(h->ev[0], s);
  ++h->n_launches;
  k_frame_reset<<<1, 1, 0, s>>>(h->d_cnt, in.d_depth ? 0 : cap);
  if (in.d_depth) {
    ++h->n_launches;
    k_depth_flags<<<grid_for(cap, B), B, 0, s>>>(in.d_depth, cap, h->flags8);
    size_t tb = h->cub_temp_bytes;
    ++h->n_libcalls;
    KSG_CUDA(cub::DeviceSelect::Flagged(h->cub_temp, tb, cub::CountingInputIterator<int>(0), h->flags8, h->pix_list,
                                        &h->d_cnt->n_points, cap, s));
  }
  if (h->cfg.integration_order_mode == KSG_ORDER_SORTED) {
    ++h->n_launches;
    k_sqnorm<<<grid_for(cap, B), B, 0, s>>>(fin, h->d_cnt, cap, h->sq_keys);
    size_t tb = h->cub_temp_bytes;
    ++h->n_libcalls;
    KSG_CUDA(cub::DeviceRadixSort::SortPairs(h->cub_temp, tb, h->sq_keys, h->sq_keys_out, h->iota, (uint32_t*)h->point_of_seq,
                                             cap, 0, 32, s));
    fin.point_of_seq = h->point_of_seq;
  }

  // ApproxHashSet resets (fast.cpp:165-170, A.4)
  if (fast) {
    if ((++h->reset_counter) >= h->cfg.clear_checks_every_n_frames) {
      h->reset_counter = 0;
      if (++h->set_offset >= 10000) {
        h->set_offset = 0;
        KSG_CUDA(cudaMemsetAsync(h->start_table, 0xFF, sizeof(uint32_t) * kSetSize, s));
        KSG_CUDA(cudaMemsetAsync(h->ob.table, 0xFF, sizeof(uint32_t) * kSetSize, s));
      }
    }
  }

  long long n_records = 0;
  int iterations = 0;
  int64_t last_hot_voxels = 0;
  ApplySrc src{};
  if (fast) {
    KSG_CUDA(cudaMemsetAsync(h->clear_ff, 0xFF, (size_t)kSetSize * 16, s));
    KSG_CUDA(cudaMemsetAsync(h->clear_00, 0x00, (size_t)kSetSize * 5, s));
    KSG_CUDA(cudaMemsetAsync(h->start_min, 0x7F, sizeof(int) * kSetSize, s));
    ++h->n_launches;
    k_classify<true><<<grid_for(cap, B), B, 0, s>>>(dc, T, fin, h->d_luts, h->set_offset, cap, h->d_cnt, h->pt_pC, h->pt_pG,
                                                    h->pt_label, h->pt_flags, h->pt_color, h->pt_key);
    ++h->n_launches;
    StartBuf sbuf{h->start_head, h->start_next, h->start_min, h->start_max, h->start_val, h->start_mixed, h->start_table};
    k_start_push<<<grid_for(cap, B), B, 0, s>>>(h->d_cnt, h->pt_key, sbuf);
    ++h->n_launches;
    k_start_eval<<<grid_for(cap, B), B, 0, s>>>(h->d_cnt, h->pt_key, sbuf, h->flags8, h->is_last, cap);
    ++h->n_launches;
    k_start_commit<<<grid_for(cap, B), B, 0, s>>>(h->d_cnt, h->pt_key, h->is_last, h->start_table);
    {
      size_t tb = h->cub_temp_bytes;
      ++h->n_libcalls;
      KSG_CUDA(cub::DeviceSelect::Flagged(h->cub_temp, tb, cub::CountingInputIterator<int>(0), h->flags8, h->cast_seq,
                                          &h->d_cnt->n_cast, cap, s));
    }
    ++h->n_launches;
    k_ray_setup<<<grid_for(cap, 128), 128, 0, s>>>(dc, T, h->d_cnt, h->cast_seq, h->pt_pG, h->pt_label, h->pt_flags, h->pt_color,
                                                   h->set_offset, h->ob, h->ray_param, h->ray_label, h->ray_flags, h->ray_color,
                                                   h->nsteps, h->H, h->L, h->ray_state, h->eval_sweep);
    if (h->profiling) cudaEventRecord(h->ev[1], s);
    // observed-set fixpoint: sweeps until no ray changes; two sweeps per host read-back
    int n_cast = cap;
    if (h->sweep_counter > 0x3FFFFFFF) {  // keep sweep ids monotonic: restart the stamps long before int overflow
      KSG_CUDA(cudaMemsetAsync(h->ob.slot_stamp, 0, sizeof(int) * kSetSize, s));
      h->sweep_counter = 0;
    }
    h->sweep_counter = (h->sweep_counter + 4) & ~3;  // counters of the first sweep (index 1) were zeroed by k_frame_reset
    if (h->persistent_eval) {
      // one cooperative launch sweeps to convergence on the device (grid barrier between sweeps)
      const int first_sweep = h->sweep_counter + 1;
      int max_sweeps = 4096;
      KSG_CUDA(cudaMemsetAsync(h->d_gridbar, 0, sizeof(unsigned int), s));
      ++h->n_launches;
      void* args[] = {(void*)&dc, (void*)&h->d_cnt, (void*)&h->set_offset, (void*)&h->ob, (void*)&h->nsteps, (void*)&h->H, (void*)&h->L,
                      (void*)&h->ray_state, (void*)&h->ext_off, (void*)&h->eval_sweep, (void*)&first_sweep, (void*)&max_sweeps, (void*)&h->d_gridbar};
      KSG_CUDA(cudaLaunchCooperativeKernel((const void*)k_eval_persistent, dim3(h->eval_grid), dim3(256), args, 0, s));
      int rc = fetch_counters(h, s);
      if (rc) return rc;
      const int last = h->h_cnt->last_sweep;
      iterations = last - first_sweep + 1;
      h->sweep_counter = last;
      n_cast = std::max(1, h->h_cnt->n_cast);
      if (!h->h_cnt->err) {
        if (h->h_cnt->changed[last & 3]) { h->deferred_status = KSG_ERR_CUDA; return fail(KSG_ERR_CUDA, "observed-set solver did not converge within 4096 sweeps"); }
        n_records = (long long)h->h_cnt->sum_updates[last & 3];
      }
    } else
    for (;;) {
      int sweep = 0;
      const int batch = (iterations == 0) ? h->first_batch : h->sweeps_per_sync;
      for (int rep = 0; rep < batch; ++rep) {
        sweep = ++h->sweep_counter;
        h->n_launches += 1;
        k_eval<<<h->sm_count * 8, 256, 0, s>>>(dc, h->d_cnt, h->set_offset, h->ob, h->nsteps, h->H, h->L, h->ray_state, h->ext_off,
                                               h->eval_sweep, sweep);
        ++iterations;
      }
      int rc = fetch_counters(h, s);
      if (rc) return rc;
      n_cast = std::max(1, h->h_cnt->n_cast);
      if (h->h_cnt->err) break;
      if (iterations > 4096) {  // theory: <= rays + 1 sweeps, practice ~10; never hang the caller
        h->deferred_status = KSG_ERR_CUDA;
        return fail(KSG_ERR_CUDA, "observed-set solver did not converge within 4096 sweeps");
      }
      if (h->h_cnt->changed[sweep & 3]) continue;
      n_records = (long long)h->h_cnt->sum_updates[sweep & 3];
      break;
    }
    if (h->profiling) cudaEventRecord(h->ev[2], s);
    if (!h->h_cnt->err) {
      if (n_records > h->rec_cap) { h->deferred_status = KSG_ERR_SCRATCH_FULL; return fail(KSG_ERR_SCRATCH_FULL, err_text(4)); }
      h->n_launches += 2;
      k_obs_commit<<<grid_for((long long)n_cast * kEvalGroup, 128), 128, 0, s>>>(h->d_cnt, h->ob, h->L, h->ext_off);
      k_emit_fast<<<grid_for(n_cast, 128), 128, 0, s>>>(dc, T, h->d_cnt, h->map, h->ray_param, h->ray_flags, h->L, h->rec_a,
                                                        h->rec_cap);
    }
    src.param = h->ray_param; src.label = h->ray_label; src.color = h->ray_color; src.tmp = nullptr;
  } else {
    ++h->n_launches;
    k_classify<false><<<grid_for(cap, B), B, 0, s>>>(dc, T, fin, h->d_luts, 0ull, cap, h->d_cnt, h->pt_pC, h->pt_pG, h->pt_label,
                                                     h->pt_flags, h->pt_color, h->pt_key);
    if (h->profiling) cudaEventRecord(h->ev[1], s);
    {
      size_t tb = h->cub_temp_bytes;
      ++h->n_libcalls;
      KSG_CUDA(cub::DeviceRadixSort::SortPairs(h->cub_temp, tb, h->pt_key, h->ks_sorted, h->iota, h->seq_sorted, cap, 0, 64, s));
    }
    KSG_CUDA(cudaMemsetAsync(h->flags8, 0, 2 * (size_t)cap, s));
    ++h->n_launches;
    k_bundle_heads<<<grid_for(cap, B), B, 0, s>>>(h->ks_sorted, h->seq_sorted, cap, h->flags8, h->bstart);
    {
      size_t tb = h->cub_temp_bytes;
      ++h->n_libcalls;
      KSG_CUDA(cub::DeviceSelect::Flagged(h->cub_temp, tb, cub::CountingInputIterator<int>(0), h->flags8, h->bundle_f,
                                          &h->d_cnt->n_cast, 2 * cap, s));
    }
    const int* bundle_heads = h->bundle_f;   // canonical: first-insertion order
    if (h->cfg.merged_bundle_order == KSG_BUNDLE_ORDER_LIBSTDCXX) {
      h->n_launches += 2;
      k_bord_hash<<<grid_for(cap, B), B, 0, s>>>(h->d_cnt, h->bundle_f, h->bstart, h->ks_sorted, cap, h->bord_hash);
      // every rehash phase of both maps (voxel_map merged.cpp:126-134, clear_map :138-145) in one launch: one cluster per map
      k_bundle_order<<<2 * kBordCluster, kBordThreads, 0, s>>>(h->d_cnt, h->bord, h->bundle_f, h->bundle_f2);
      bundle_heads = h->bundle_f2;
    }
    ++h->n_launches;
    k_bundle_merge<<<h->sm_count * 8, 256, 0, s>>>(dc, T, h->d_cnt, bundle_heads, h->bstart, h->ks_sorted, h->seq_sorted, cap, h->pt_pC,
                                                   h->pt_label, h->hist, h->ray_param, h->ray_flags, h->b_key, h->nsteps);
    ++h->n_launches;
    k_bundle_scan<<<kBordCluster, kBordThreads, 0, s>>>(h->d_cnt, h->nsteps, h->b_base, h->rec_cap, h->d_scan_tot);
    int rc = fetch_counters(h, s);
    if (rc) return rc;
    if (h->profiling) cudaEventRecord(h->ev[2], s);
    if (!h->h_cnt->err) {
      const int nb = std::max(1, h->h_cnt->n_cast);
      n_records = (long long)h->h_cnt->n_records;
      ++h->n_launches;
      k_bundle_loglik<<<grid_for((long long)(nb + 1) * dc.C, B), B, 0, s>>>(dc, h->d_cnt, h->hist, h->tmp, h->tmp4);
      ++h->n_launches;
      if (h->emit_warp)
        k_emit_merged_warp<<<h->sm_count * 8, 256, 0, s>>>(dc, T, h->d_cnt, h->map, h->ray_param, h->ray_flags, h->b_key, h->nsteps, h->b_base,
                                                           h->ks_sorted, cap, h->rec_a);
      else
      k_emit_merged<<<grid_for(nb, 128), 128, 0, s>>>(dc, T, h->d_cnt, h->map, h->ray_param, h->ray_flags, h->b_key, h->nsteps,
                                                      h->b_base, h->ks_sorted, cap, h->rec_a);
    }
    src.param = h->ray_param; src.label = nullptr; src.color = nullptr; src.tmp = h->tmp; src.tmp4 = h->tmp4;
  }

  if (h->profiling) cudaEventRecord(h->ev[3], s);
  int dev_err = h->h_cnt->err;
  bool did_apply = false;
  if (!dev_err && n_records > 0) {
    // order the update records by (tile, voxel, order): per-voxel application order = reference order
    size_t tb = h->cub_temp_bytes;
    ++h->n_libcalls;
    // significant key bits: [order 23][voxel 9][tile key < ht_cap * tiles_per_block]
    int end_bit = 32;
    while (end_bit < 64 && (1ull << (end_bit - 32)) < (unsigned long long)h->ht_cap * (unsigned long long)dc.tiles_per_block) ++end_bit;
    // merged: the records were laid out by (bundle rank, step), so a stable sort on the voxel bits [23, end) keeps the rank order
    KSG_CUDA(cub::DeviceRadixSort::SortKeys(h->cub_temp, tb, h->rec_a, h->rec_b, n_records, fast ? 0 : kRecOrdBits, end_bit, s));
    if (h->profiling) cudaEventRecord(h->ev[4], s);
    ++h->n_launches;
    k_block_init<<<h->sm_count * 4, 256, 0, s>>>(dc, h->d_cnt, h->map);
    if (h->voxel_apply && !fast) {
      // per-voxel update (ksg_voxel.cuh): segment heads -> two queues; the long and the short kernel run concurrently
      KSG_CUDA(cudaMemsetAsync(h->vq.counters, 0, sizeof(int) * 8, s));
      ++h->n_launches;
      k_voxel_heads<<<grid_for(n_records, kHeadsBlock), 256, 0, s>>>(dc, h->d_cnt, h->map, h->rec_b, n_records, h->frame_stamp, h->vq);
      if (h->profiling) cudaEventRecord(h->ev[5], s);
      did_apply = true;
      if (h->hot_enabled) {
        int n_hot = 0;
        const int rch = hot_voxel_prepass(h, s, T, src.param, n_records, &n_hot);
        if (rch) return rch;
        src.hot_segs = h->d_hot_segs; src.hot_prior = h->d_hot_prior; src.n_hot = n_hot; src.hot_thresh = kHotThresh;
        src.hot_tsdf_same = (h->cfg.hot_voxel_mode == 2) ? h->d_hot_same : nullptr;
        last_hot_voxels = n_hot;
      }
      KSG_CUDA(cudaEventRecord(h->ev_fork, s));
      KSG_CUDA(cudaStreamWaitEvent(h->aux_stream, h->ev_fork, 0));
      // C <= 32: the voxels with thousands of records get one CTA each (third stream, concurrent with the other two kernels)
      const int use_hot = (h->apply_nch == 1 && !h->hot_enabled && h->hot_kernel) ? 1 : 0;
      bool deep_launched = false;
      if (use_hot) {
        KSG_CUDA(cudaStreamWaitEvent(h->aux_stream2, h->ev_fork, 0));
        ++h->n_launches;
        k_voxel_apply_hot<<<h->sm_count, 256, h->hot_smem, h->aux_stream2>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, src, h->vq);
        KSG_CUDA(cudaEventRecord(h->ev_join2, h->aux_stream2));
      }
      h->n_launches += 2;
#define KSG_LAUNCH_VOXEL(NCH)                                                                                                             \
      do {                                                                                                                                \
        k_voxel_apply_long<NCH><<<h->long_grid, h->long_threads, 0, h->aux_stream>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, src, h->vq, use_hot);  \
        k_voxel_apply_short<NCH><<<h->sm_count * h->short_ctas, 256, h->short_smem, s>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, src, h->vq);        \
      } while (0)
      if (h->short_thread && h->apply_nch == 1) {
        int skip = use_hot;
        if (h->deep_hot && !use_hot) {   // the hot voxels' chains first, on their own high-priority stream (one warp per chain)
          KSG_CUDA(cudaStreamWaitEvent(h->aux_stream2, h->ev_fork, 0));
          ++h->n_launches;
          k_voxel_apply_long<1, true><<<h->sm_count, h->deep_threads, 0, h->aux_stream2>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, src, h->vq, 0);
          KSG_CUDA(cudaEventRecord(h->ev_join2, h->aux_stream2));
          skip = 1; deep_launched = true;
        }
        if (h->long_serial && deep_launched) {   // the remaining long segments are little work: behind the short kernel, on its stream
          k_voxel_apply_short_t<<<h->sm_count * h->short_t_ctas, 256, 0, s>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, src, h->vq);
          k_voxel_apply_long<1><<<h->long_grid, h->long_threads, 0, s>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, src, h->vq, skip);
        } else {
          k_voxel_apply_long<1><<<h->long_grid, h->long_threads, 0, h->aux_stream>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, src, h->vq, skip);
          k_voxel_apply_short_t<<<h->sm_count * h->short_t_ctas, 256, 0, s>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, src, h->vq);
        }
      } else
      switch (h->apply_nch) { case 1: KSG_LAUNCH_VOXEL(1); break; case 2: KSG_LAUNCH_VOXEL(2); break; case 4: KSG_LAUNCH_VOXEL(4); break; default: KSG_LAUNCH_VOXEL(8); break; }
#undef KSG_LAUNCH_VOXEL
      KSG_CUDA(cudaEventRecord(h->ev_join, h->aux_stream));
      KSG_CUDA(cudaStreamWaitEvent(s, h->ev_join, 0));
      if (use_hot || deep_launched) KSG_CUDA(cudaStreamWaitEvent(s, h->ev_join2, 0));
    } else {
    ++h->n_launches;
    k_tile_heads<<<grid_for(n_records, B), B, 0, s>>>(dc, h->d_cnt, h->map, h->rec_b, n_records, h->frame_stamp, h->tile_begin,
                                                      h->tile_cap);

    if (h->profiling) cudaEventRecord(h->ev[5], s);
    did_apply = true;
    const int ctas_per_sm = std::max(1, std::min(8, (int)(220 * 1024 / std::max(1, h->apply_smem + 1024))));
    const int grid = h->sm_count * ctas_per_sm;
    const int apply_threads = fast ? 512 : 256;  // fast: few records per voxel, latency bound -> more warps per tile
    int n_hot = 0;
    if (h->hot_enabled) {
      const int rch = hot_voxel_prepass(h, s, T, src.param, n_records, &n_hot);
      if (rch) return rch;
      src.hot_segs = h->d_hot_segs; src.hot_prior = h->d_hot_prior; src.n_hot = n_hot; src.hot_thresh = kHotThresh;
      src.hot_tsdf_same = (h->cfg.hot_voxel_mode == 2) ? h->d_hot_same : nullptr;
      last_hot_voxels = n_hot;
    }
    ++h->n_launches;
    if (n_hot > 0) {   // merged, C <= 32, TMA staging (checked when hot_enabled was set)
      k_tile_apply<true, 1, true, true><<<grid, apply_threads, h->apply_smem, s>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, n_records,
                                                                                  h->tile_begin, h->tile_cap, src, h->tile_debug);
    } else
#define KSG_LAUNCH_APPLY_(TMA, NCH, MRG)                                                                                 \
    k_tile_apply<TMA, NCH, MRG><<<grid, apply_threads, h->apply_smem, s>>>(dc, T, h->d_cnt, h->map, h->d_luts, h->rec_b, \
                                                                      n_records, h->tile_begin, h->tile_cap, src, h->tile_debug)
#define KSG_LAUNCH_APPLY(TMA, NCH) do { if (fast) { KSG_LAUNCH_APPLY_(TMA, NCH, false); } else { KSG_LAUNCH_APPLY_(TMA, NCH, true); } } while (0)
    if (h->use_tma) {
      switch (h->apply_nch) { case 1: KSG_LAUNCH_APPLY(true, 1); break; case 2: KSG_LAUNCH_APPLY(true, 2); break;
                              case 4: KSG_LAUNCH_APPLY(true, 4); break; default: KSG_LAUNCH_APPLY(true, 8); break; }
    } else {
      switch (h->apply_nch) { case 1: KSG_LAUNCH_APPLY(false, 1); break; case 2: KSG_LAUNCH_APPLY(false, 2); break;
                              case 4: KSG_LAUNCH_APPLY(false, 4); break; default: KSG_LAUNCH_APPLY(false, 8); break; }
    }
#undef KSG_LAUNCH_APPLY_
#undef KSG_LAUNCH_APPLY
    }
  }
  if (h->profiling) { if (!did_apply) { cudaEventRecord(h->ev[4], s); cudaEventRecord(h->ev[5], s); } cudaEventRecord(h->ev[6], s); }
  ++h->n_launches;
  k_frame_finish<<<1, 1, 0, s>>>(h->d_cnt, h->map);
  KSG_CUDA(cudaGetLastError());
  int rc = fetch_counters(h, s);
  if (rc) return rc;
  if (h->profiling) {
    cudaEventRecord(h->ev[7], s);
    cudaEventSynchronize(h->ev[7]);
    for (int p = 0; p < 6; ++p) { float ms = 0; if (cudaEventElapsedTime(&ms, h->ev[p], h->ev[p + 1]) == cudaSuccess) h->phase_ms[p] += ms; }
    { float ms = 0; if (cudaEventElapsedTime(&ms, h->ev[0], h->ev[7]) == cudaSuccess) h->phase_ms[6] += ms; }
    h->prof_frames += 1;
  }
  dev_err = h->h_cnt->err;
  h->num_blocks = h->h_cnt->pool_count;
  h->last_blocks_touched = h->h_cnt->n_blocks_touched;
  if (stats) {
    std::memset(stats, 0, sizeof(*stats));
    stats->points_in = h->h_cnt->n_points;
    stats->points_valid = h->h_cnt->n_valid;
    stats->rays_cast = h->h_cnt->n_cast;
    stats->ray_steps = (int64_t)h->h_cnt->ray_steps;
    stats->voxel_updates = n_records - (int64_t)h->h_cnt->n_skipped;
    stats->blocks_allocated = h->num_blocks;
    stats->blocks_touched = h->h_cnt->n_blocks_touched;
    stats->tiles_touched = h->h_cnt->n_tiles;
    stats->fixpoint_iterations = iterations;
    stats->hot_voxels = last_hot_voxels;
    if (h->hot_enabled && last_hot_voxels > 0) {
      int fb = 0;
      if (cudaMemcpyAsync(&fb, h->d_hot_counts + 1, sizeof(int), cudaMemcpyDeviceToHost, s) == cudaSuccess && cudaStreamSynchronize(s) == cudaSuccess)
        stats->hot_fallback_chunks = fb;
    }
  }
  if (dev_err) {
    h->deferred_status = dev_err;  // the map may be inconsistent from here on
    return fail(dev_err, err_text(dev_err));
  }
  return KSG_OK;
}

bool is_pinned_host(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

int ensure_input(ksg_integrator* h, size_t bytes) {
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  if (bytes > h->h_stage_bytes) {
    if (h->h_stage) cudaFreeHost(h->h_stage);
    h->h_stage = nullptr;
    KSG_CUDA(cudaMallocHost((void**)&h->h_stage, bytes));
    h->h_stage_bytes = bytes;
  }
  if (bytes > h->d_in_bytes) {
    if (h->d_in) cudaFree(h->d_in);
    h->d_in = nullptr;
    KSG_CUDA(cudaMalloc((void**)&h->d_in, bytes));
    h->d_in_bytes = bytes;
  }
  return KSG_OK;
}

}  // namespace

extern "C" {

void ksg_default_config(ksg_config* c, int32_t integrator_type, float voxel_size, int32_t voxels_per_side, int32_t num_labels) {
  std::memset(c, 0, sizeof(*c));
  c->abi_version = KSG_ABI_VERSION;
  c->integrator_type = integrator_type;
  c->voxel_size = voxel_size;
  c->voxels_per_side = voxels_per_side;
  c->default_truncation_distance = 4.0f * voxel_size;  // voxblox_ros: truncation_distance = 4 * voxel_size
  c->max_weight = 10000.0f;
  c->voxel_carving_enabled = 1;
  c->min_ray_length_m = 0.1f;
  c->max_ray_length_m = 5.0f;
  c->use_const_weight = 0;
  c->allow_clear = 1;
  c->use_weight_dropoff = 1;
  c->use_sparsity_compensation_factor = 0;
  c->sparsity_compensation_factor = 1.0f;
  c->integration_order_mode = KSG_ORDER_MIXED;
  c->enable_anti_grazing = 0;
  c->start_voxel_subsampling_factor = 2.0f;
  c->max_consecutive_ray_collisions = 2;
  c->clear_checks_every_n_frames = 1;
  c->integrator_threads = 1;
  c->num_labels = num_labels;
  c->semantic_measurement_probability = 0.9f;  // base.h:77
  c->color_mode = KSG_COLOR_MODE_SEMANTIC;     // base.h:80
  for (int l = 0; l < 256; ++l) {
    c->label_color[l][0] = 127; c->label_color[l][1] = 127; c->label_color[l][2] = 127; c->label_color[l][3] = 255;
    c->label_color_known[l] = 1;
    c->dynamic_label[l] = 0;
  }
  c->device = 0;
  c->max_blocks = 8192;
  c->max_points = 640 * 480;
  c->max_ray_steps = 0;
  c->max_updates = 0;
  c->apply_mode = 0;
  c->shard_rank = 0;
  c->shard_count = 1;
  c->merged_bundle_order = KSG_BUNDLE_ORDER_LIBSTDCXX;   // the reference's unordered_map iteration order (merged.cpp:210-231)
  c->hot_voxel_mode = 0;   // opt-in (measured slower than the per-voxel kernels alone, profiles/r02/bench_merged2_hot.json)
}

#define KSG_STR_(x) #x
#define KSG_STR(x) KSG_STR_(x)
const char* ksg_build_info(void) { return "ksg abi " KSG_STR(KSG_ABI_VERSION) " sm_100a nvcc " KSG_STR(__CUDACC_VER_MAJOR__) "." KSG_STR(__CUDACC_VER_MINOR__) " built " __DATE__; }

const char* ksg_last_error(const ksg_integrator* h) { return h ? h->err.c_str() : g_last_error.c_str(); }

int32_t ksg_create(const ksg_config* cfg, ksg_integrator** out) {
  if (!out) return KSG_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  std::string why;
  int rc = validate(cfg, why);
  if (rc) { g_last_error = why; return rc; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || cfg->device >= ndev) {
    g_last_error = "no CUDA device (the integrator has no CPU fallback)";
    cudaGetLastError();
    return KSG_ERR_NO_DEVICE;
  }
  ksg_integrator* h = new ksg_integrator();
  h->cfg = *cfg;
  h->device = cfg->device;
  auto fail = [&](int c, const char* m) { g_last_error = m; free_all(h); delete h; return c; };
  KSG_CUDA(cudaSetDevice(h->device));
  cudaDeviceProp prop;
  KSG_CUDA(cudaGetDeviceProperties(&prop, h->device));
  h->sm_count = prop.multiProcessorCount;
  KSG_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));

  // ---- geometry (voxblox Layer: inverses are 1.0 / x in double, stored as float; A.1, base.cpp:84-89)
  DevCfg& dc = h->dc;
  dc.voxel_size = cfg->voxel_size;
  dc.vsi = (float)(1.0 / cfg->voxel_size);
  dc.vps = cfg->voxels_per_side;
  dc.vps_inv = (float)(1.0f / (float)cfg->voxels_per_side);
  dc.tile_side = std::min(cfg->voxels_per_side, kTileSideMax);
  dc.tile_side_log2 = ilog2(dc.tile_side);
  dc.tiles_per_side = dc.vps / dc.tile_side;
  dc.tiles_per_block = dc.tiles_per_side * dc.tiles_per_side * dc.tiles_per_side;
  dc.tile_voxels = dc.tile_side * dc.tile_side * dc.tile_side;
  dc.plane_f32 = round_up(4u * dc.tile_voxels, 16);
  dc.plane_u8 = round_up((uint32_t)dc.tile_voxels, 16);
  dc.head_bytes = 4 * dc.plane_f32 + dc.plane_u8;
  dc.C = cfg->num_labels;
  dc.prior_bytes = round_up(4u * (uint32_t)dc.tile_voxels * (uint32_t)dc.C, 16);
  dc.tile_stride = round_up(dc.head_bytes + dc.prior_bytes, 128);
  dc.full_stage = (dc.head_bytes + dc.prior_bytes + 8u * dc.tile_voxels + 64u) <= 72u * 1024u ? 1 : 0;
  dc.block_stride = (uint64_t)dc.tile_stride * dc.tiles_per_block;
  dc.tp.voxel_size = cfg->voxel_size;
  dc.tp.trunc = cfg->default_truncation_distance;
  dc.tp.max_weight = cfg->max_weight;
  dc.tp.sparsity_factor = cfg->sparsity_compensation_factor;
  dc.tp.use_weight_dropoff = cfg->use_weight_dropoff;
  dc.tp.use_sparsity = cfg->use_sparsity_compensation_factor;
  dc.min_ray = cfg->min_ray_length_m;
  dc.max_ray = cfg->max_ray_length_m;
  dc.start_inv = cfg->start_voxel_subsampling_factor * dc.vsi;  // fast.cpp:89
  dc.carving = cfg->voxel_carving_enabled;
  dc.const_weight = cfg->use_const_weight;
  // voxblox TsdfIntegratorBase ctor: clearing rays have no use without carving, so allow_clear is forced off there
  // (explicit freespace clouds still clear, isPointValid tests allow_clear || freespace_points)
  dc.allow_clear = (cfg->allow_clear && cfg->voxel_carving_enabled) ? 1 : 0;
  dc.maxc = cfg->max_consecutive_ray_collisions;
  dc.anti_grazing = cfg->enable_anti_grazing;
  // setSemanticProbabilities (base.cpp:93-128): std::log on float, on the host (same libm as the reference)
  dc.lm = std::log(cfg->semantic_measurement_probability);
  dc.ln = std::log(1.0f - cfg->semantic_measurement_probability);
  dc.color_mode = cfg->color_mode;
  dc.type = cfg->integrator_type;
  dc.shard_rank = cfg->shard_rank;
  dc.shard_count = cfg->shard_count > 1 ? cfg->shard_count : 1;

  // ---- look-up tables
  for (int l = 0; l < 256; ++l) {
    const uint8_t* c = cfg->label_color[l];
    h->h_luts.label_rgba[l] = cfg->label_color_known[l] ? ((uint32_t)c[0] | ((uint32_t)c[1] << 8) | ((uint32_t)c[2] << 16) | ((uint32_t)c[3] << 24)) : 0u;
    h->h_luts.dynamic_label[l] = cfg->dynamic_label[l];
  }
  for (int i = 0; i < 1024; ++i) { h->h_luts.c2l_keys[i] = 0xFFFFFFFFu; h->h_luts.c2l_vals[i] = 0; }
  KSG_CUDA(dmalloc(&h->d_luts, 1));
  KSG_CUDA(cudaMemcpy(h->d_luts, &h->h_luts, sizeof(Luts), cudaMemcpyHostToDevice));

  // ---- map
  h->ht_cap = 1024;
  while (h->ht_cap < 2u * (uint32_t)cfg->max_blocks) h->ht_cap <<= 1;
  if ((unsigned long long)h->ht_cap * dc.tiles_per_block >= (1ull << 32)) return fail(KSG_ERR_INVALID_ARGUMENT, "max_blocks too large");
  h->map.ht_mask = h->ht_cap - 1;
  h->map.max_blocks = cfg->max_blocks;
  h->map.new_cap = cfg->max_blocks;
  KSG_CUDA(dmalloc(&h->map.ht_keys, h->ht_cap));
  KSG_CUDA(dmalloc(&h->map.ht_slot, h->ht_cap));
  KSG_CUDA(dmalloc(&h->map.touched_stamp, h->ht_cap));
  KSG_CUDA(dmalloc(&h->map.touched_list, h->ht_cap));
  KSG_CUDA(dmalloc(&h->map.new_list, (size_t)cfg->max_blocks));
  KSG_CUDA(dmalloc(&h->map.slot_key, (size_t)cfg->max_blocks));
  KSG_CUDA(cudaMalloc((void**)&h->map.pool, (size_t)dc.block_stride * (size_t)cfg->max_blocks));
  KSG_CUDA(dmalloc(&h->d_cnt, 1));
  KSG_CUDA(cudaMallocHost((void**)&h->h_cnt_base, 2 * sizeof(Counters)));
  std::memset(h->h_cnt_base, 0, 2 * sizeof(Counters));
  h->h_cnt = h->h_cnt_base;
  for (int i = 0; i < 2; ++i) {
    KSG_CUDA(cudaEventCreateWithFlags(&h->ev_frame_s[i], cudaEventDisableTiming));
    KSG_CUDA(cudaEventCreateWithFlags(&h->ev_copy[i], cudaEventDisableTiming));
    KSG_CUDA(cudaEventCreateWithFlags(&h->ev_free[i], cudaEventDisableTiming));
  }
  KSG_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));

  // ---- frame scratch
  const size_t N = (size_t)cfg->max_points;
  h->cap_points = cfg->max_points;
  const bool fast = cfg->integrator_type == KSG_INTEGRATOR_FAST;
  KSG_CUDA(dmalloc(&h->pt_pC, N)); KSG_CUDA(dmalloc(&h->pt_pG, N));
  KSG_CUDA(dmalloc(&h->pt_label, N)); KSG_CUDA(dmalloc(&h->pt_flags, N));
  KSG_CUDA(dmalloc(&h->pt_color, N)); KSG_CUDA(dmalloc(&h->pt_key, N));
  KSG_CUDA(dmalloc(&h->flags8, 2 * N)); KSG_CUDA(dmalloc(&h->is_last, N));
  KSG_CUDA(dmalloc(&h->pix_list, N));
  KSG_CUDA(dmalloc(&h->iota, N));
  k_iota<<<grid_for((long long)N, 256), 256>>>(h->iota, (int)N);
  if (cfg->integration_order_mode == KSG_ORDER_SORTED) {
    KSG_CUDA(dmalloc(&h->point_of_seq, N)); KSG_CUDA(dmalloc(&h->sq_keys, N)); KSG_CUDA(dmalloc(&h->sq_keys_out, N));
  }
  KSG_CUDA(dmalloc(&h->ray_param, N)); KSG_CUDA(dmalloc(&h->ray_flags, N)); KSG_CUDA(dmalloc(&h->nsteps, N));
  long long rec_cap = cfg->max_updates > 0 ? cfg->max_updates : (fast ? std::max<long long>(4ll << 20, 64ll * (long long)N) : (64ll << 20));
  if (fast) {
    KSG_CUDA(dmalloc(&h->start_next, N)); KSG_CUDA(dmalloc(&h->start_table, kSetSize));
    // per-frame cleared arrays live in two contiguous regions: [0xFF: start_head | start_max | start_val | ob.head] and
    // [0x00: ob.slot_cnt | start_mixed], so that a frame needs three memsets instead of seven
    KSG_CUDA(cudaMalloc((void**)&h->clear_ff, (size_t)kSetSize * 16));
    KSG_CUDA(cudaMalloc((void**)&h->clear_00, (size_t)kSetSize * 13));   // [ob.slot_cnt 4 | start_mixed 1 | s_hmax 4 | s_visits 4] bytes per slot
    h->start_head = (int*)h->clear_ff; h->start_max = h->start_head + kSetSize; h->start_val = (uint32_t*)(h->start_max + kSetSize);
    h->start_mixed = h->clear_00 + (size_t)kSetSize * 4;
    KSG_CUDA(dmalloc(&h->start_min, kSetSize));
    KSG_CUDA(dmalloc(&h->cast_seq, N));
    KSG_CUDA(dmalloc(&h->ray_label, N)); KSG_CUDA(dmalloc(&h->ray_color, N));
    KSG_CUDA(dmalloc(&h->H, N)); KSG_CUDA(dmalloc(&h->L, N)); KSG_CUDA(dmalloc(&h->ray_state, N)); KSG_CUDA(dmalloc(&h->ext_off, N * kExtSegs));
    KSG_CUDA(dmalloc(&h->eval_sweep, N)); KSG_CUDA(dmalloc(&h->ob.slot_stamp, kSetSize));
    long long ext = cfg->max_ray_steps > 0 ? cfg->max_ray_steps : std::max<long long>(16ll << 20, 64ll * (long long)N);
    h->ob.ext_base = (long long)N * kH0;
    h->ob.cand_cap = h->ob.ext_base + ext;
    if (h->ob.cand_cap >= 0x7FFFFFFFll) { h->ob.cand_cap = 0x7FFFFFFEll; }
    {
      bool legacy = false;
      if (const char* e = std::getenv("KSG_FAST_LEGACY")) legacy = std::atoi(e) != 0;
      if (const char* e = std::getenv("KSG_SOLVER")) h->solver = (std::atoi(e) == 2) ? 2 : 3;
      if (legacy || h->solver == 2) {
        KSG_CUDA(dmalloc(&h->ob.cand_val, (size_t)h->ob.cand_cap)); KSG_CUDA(dmalloc(&h->ob.cand_order, (size_t)h->ob.cand_cap));
        KSG_CUDA(dmalloc(&h->ob.cand_next, (size_t)h->ob.cand_cap)); KSG_CUDA(dmalloc(&h->ob.cand_pos, (size_t)h->ob.cand_cap));
      } else {
        KSG_CUDA(cudaMalloc((void**)&h->cand16, sizeof(Cand) * (size_t)h->ob.cand_cap));
        h->ovf_cap = (int)std::min<long long>(std::max<long long>(1ll << 20, 4ll * (long long)N), 1ll << 28);
        KSG_CUDA(cudaMalloc((void**)&h->ovf, sizeof(OvfEnt) * (size_t)h->ovf_cap));
        KSG_CUDA(cudaMalloc((void**)&h->rayrec, sizeof(RayRec) * N));
        KSG_CUDA(dmalloc(&h->mixed_list, N)); KSG_CUDA(dmalloc(&h->m_list, N));
        KSG_CUDA(dmalloc(&h->blk_run, (size_t)(h->ob.cand_cap / 16 + 16)));
        KSG_CUDA(dmalloc(&h->stamp64, 2 * (size_t)kSetSize));
      }
    }
    h->ob.slot_cnt = (int*)h->clear_00; KSG_CUDA(dmalloc(&h->ob.bkt, (size_t)kSetSize * (kBkt3 > kBktK ? kBkt3 : kBktK)));
    h->ob.head = (int*)(h->clear_ff + (size_t)kSetSize * 12); KSG_CUDA(dmalloc(&h->ob.table, kSetSize));
  } else {
    KSG_CUDA(dmalloc(&h->ks_sorted, N)); KSG_CUDA(dmalloc(&h->seq_sorted, N));
    KSG_CUDA(dmalloc(&h->bstart, 2 * N)); KSG_CUDA(dmalloc(&h->bundle_f, N));
    KSG_CUDA(dmalloc(&h->hist, N * dc.C)); KSG_CUDA(dmalloc(&h->tmp, (N + 1) * dc.C));  // + the all-zero row
    KSG_CUDA(dmalloc(&h->b_key, N)); KSG_CUDA(dmalloc(&h->b_base, N));
    KSG_CUDA(dmalloc(&h->d_scan_tot, 16));
    // per-voxel apply kernels (default); the tile kernel stays for apply_mode 1 and KSG_MERGED_TILE_APPLY=1
    h->voxel_apply = cfg->apply_mode == 0;
    if (const char* e = std::getenv("KSG_MERGED_TILE_APPLY")) if (std::atoi(e) != 0) h->voxel_apply = false;
    if (h->voxel_apply) {
      h->vq.long_cap = 4 * (rec_cap / kLongLen) + 64;
      h->vq.long_len = kLongLen;
      if (dc.C <= 32) {   // one thread per short voxel (ksg_voxel.cuh); KSG_SHORT_THREAD=0 selects the warp-per-voxel kernel, KSG_LONG_LEN the split
        h->short_thread = true;
        if (const char* e = std::getenv("KSG_SHORT_THREAD")) h->short_thread = std::atoi(e) != 0;
        if (h->short_thread) {
          KSG_CUDA(dmalloc(&h->tmp4, (N + 1) * (size_t)((dc.C + 3) & ~3)));
          h->vq.long_len = kLongLenThread;
          if (const char* e = std::getenv("KSG_LONG_LEN")) h->vq.long_len = std::max(kLongLen, std::min(1 << 20, std::atoi(e)));
        }
      }
      h->vq.short_cap = rec_cap;
      KSG_CUDA(dmalloc(&h->vq.long_items, (size_t)h->vq.long_cap));
      KSG_CUDA(dmalloc(&h->vq.counters, 8));
      {   // the long-segment kernel must get its CTAs placed before the short-segment kernel fills the register files: its stream has priority
        int lo_p = 0, hi_p = 0;
        KSG_CUDA(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
        KSG_CUDA(cudaStreamCreateWithPriority(&h->aux_stream, cudaStreamNonBlocking, hi_p));
      }
      KSG_CUDA(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
      KSG_CUDA(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
      {
        int lo_p = 0, hi_p = 0;
        KSG_CUDA(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
        KSG_CUDA(cudaStreamCreateWithPriority(&h->aux_stream2, cudaStreamNonBlocking, hi_p));
      }
      KSG_CUDA(cudaEventCreateWithFlags(&h->ev_join2, cudaEventDisableTiming));
      if (const char* e = std::getenv("KSG_L2_PERSIST")) {
        // experiment: keep the (L * freq) rows resident in L2 while the update kernels stream records and voxel data through it
        if (std::atoi(e) != 0) {
          cudaDeviceProp prop{};
          KSG_CUDA(cudaGetDeviceProperties(&prop, h->device));
          const size_t want = std::min<size_t>((size_t)prop.persistingL2CacheMaxSize, 32u << 20);
          if (want > 0) {
            KSG_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want));
            cudaStreamAttrValue attr{};
            attr.accessPolicyWindow.base_ptr = h->tmp;
            attr.accessPolicyWindow.num_bytes = std::min<size_t>((size_t)(N + 1) * dc.C * sizeof(float), (size_t)prop.accessPolicyMaxWindowSize);
            attr.accessPolicyWindow.hitRatio = 1.0f;
            attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            KSG_CUDA(cudaStreamSetAttribute(h->aux_stream2, cudaStreamAttributeAccessPolicyWindow, &attr));
            KSG_CUDA(cudaStreamSetAttribute(h->aux_stream, cudaStreamAttributeAccessPolicyWindow, &attr));
          }
        }
      }
      h->hot_smem = 2 * kHotChunkRecs * (32 * (int)sizeof(float) + (int)sizeof(float4));
      KSG_CUDA(cudaFuncSetAttribute(k_voxel_apply_hot, cudaFuncAttributeMaxDynamicSharedMemorySize, h->hot_smem));
      if (const char* e = std::getenv("KSG_HOT_KERNEL")) h->hot_kernel = std::atoi(e) != 0;
      h->long_grid = h->sm_count;
      if (const char* e = std::getenv("KSG_LONG_THREADS")) { const int t = std::atoi(e); if (t == 64 || t == 128 || t == 256) h->long_threads = t; }
      if (const char* e = std::getenv("KSG_LONG_GRID")) h->long_grid = std::max(1, std::atoi(e));
      if (const char* e = std::getenv("KSG_DEEP_HOT")) h->deep_hot = std::atoi(e) != 0;
      if (const char* e = std::getenv("KSG_LONG_SERIAL")) h->long_serial = std::atoi(e) != 0;
      if (const char* e = std::getenv("KSG_DEEP_THREADS")) { const int t = std::atoi(e); if (t == 32 || t == 64 || t == 128 || t == 256) h->deep_threads = t; }
      if (const char* e = std::getenv("KSG_SHORT_T_CTAS")) h->short_t_ctas = std::max(1, std::min(8, std::atoi(e)));
      if (const char* e = std::getenv("KSG_SHORT_CTAS")) h->short_ctas = std::max(1, std::min(6, std::atoi(e)));
      if (h->short_ctas < 6) {
        h->short_smem = std::min(200 * 1024, (220 * 1024) / h->short_ctas - 2048);
        KSG_CUDA(cudaFuncSetAttribute(k_voxel_apply_short<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->short_smem));
        KSG_CUDA(cudaFuncSetAttribute(k_voxel_apply_short<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->short_smem));
        KSG_CUDA(cudaFuncSetAttribute(k_voxel_apply_short<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->short_smem));
        KSG_CUDA(cudaFuncSetAttribute(k_voxel_apply_short<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->short_smem));
      }
      if (const char* e = std::getenv("KSG_EMIT_WARP")) h->emit_warp = std::atoi(e) != 0;
    }
    if (cfg->hot_voxel_mode >= 1 && dc.C <= 32 && cfg->apply_mode == 0) {
      h->hot_enabled = true;
      h->hot_chunk_cap = rec_cap / kHotChunk + kHotMaxSegs;
      KSG_CUDA(dmalloc(&h->d_hot_segs, kHotMaxSegs)); KSG_CUDA(dmalloc(&h->d_hot_counts, 2));
      KSG_CUDA(cudaMemset(h->d_hot_counts, 0, 2 * sizeof(int)));
      KSG_CUDA(cudaMallocHost((void**)&h->h_hot_segs, sizeof(HotSeg) * kHotMaxSegs));
      KSG_CUDA(cudaMallocHost((void**)&h->h_hot_chunk_seg, sizeof(int) * (size_t)h->hot_chunk_cap));
      KSG_CUDA(dmalloc(&h->d_hot_chunk_seg, (size_t)h->hot_chunk_cap)); KSG_CUDA(dmalloc(&h->d_hot_guess, (size_t)h->hot_chunk_cap * 32));
      KSG_CUDA(dmalloc(&h->d_hot_sums, (size_t)h->hot_chunk_cap * 32)); KSG_CUDA(dmalloc(&h->d_hot_tables, (size_t)h->hot_chunk_cap * 32));
      KSG_CUDA(dmalloc(&h->d_hot_prior, (size_t)kHotMaxSegs * 32)); KSG_CUDA(dmalloc(&h->d_hot_same, (size_t)kHotMaxSegs));
      KSG_CUDA(cudaFuncSetAttribute(k_hot_chunk_tables, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(float) * 32 * kHotColStride)));
    }
    if (cfg->merged_bundle_order == KSG_BUNDLE_ORDER_LIBSTDCXX) {
      // rehash schedule of the platform's libstdc++ (depends on the size only): probe a real container once
      std::unordered_map<uint64_t, char> probe;
      size_t last = 0;
      for (size_t i = 0; i < N; ++i) {
        probe.emplace((uint64_t)i, 0);
        if (probe.bucket_count() != last) { last = probe.bucket_count(); h->bord_phases.push_back(std::make_pair((int)i, (uint32_t)last)); }
      }
      if (last >= 0x7fffffffull) return fail(KSG_ERR_INVALID_ARGUMENT, "max_points too large for merged_bundle_order");
      KSG_CUDA(dmalloc(&h->bord_hash, N)); KSG_CUDA(dmalloc(&h->bundle_f2, N));
      {   // scratch of k_bundle_order: [ord_a | ord_b | next | size_at | rank : N each][first | head : 2 * last each][cta_tot][phase tables]
        const size_t np = h->bord_phases.size();
        const size_t ints = 5 * N + 4 * last + 2 * kBordCluster + 2 * np + 64;
        KSG_CUDA(dmalloc(&h->bord_scratch, ints));
        int* p = h->bord_scratch;
        BordBuf& bb = h->bord;
        bb.hash = h->bord_hash;
        bb.ord_a = p; p += N; bb.ord_b = p; p += N; bb.next = p; p += N; bb.size_at = p; p += N; bb.rank = p; p += N;
        bb.first = p; p += 2 * last; bb.head = p; p += 2 * last; bb.cta_tot = p; p += 2 * kBordCluster;
        bb.bucket_cap = (uint32_t)last;
        bb.n_phases = (int)np;
        std::vector<int> ps(np); std::vector<uint32_t> pb(np);
        for (size_t i = 0; i < np; ++i) { ps[i] = h->bord_phases[i].first; pb[i] = h->bord_phases[i].second; }
        KSG_CUDA(cudaMemcpy(p, ps.data(), sizeof(int) * np, cudaMemcpyHostToDevice)); bb.phase_start = p; p += np;
        KSG_CUDA(cudaMemcpy(p, pb.data(), sizeof(uint32_t) * np, cudaMemcpyHostToDevice)); bb.phase_buckets = (const uint32_t*)p;
      }
    }
  }
  h->rec_cap = rec_cap;
  KSG_CUDA(dmalloc(&h->rec_a, (size_t)rec_cap)); KSG_CUDA(dmalloc(&h->rec_b, (size_t)rec_cap));
  h->vq.short_items = (unsigned long long*)h->rec_a;   // the unsorted record buffer is free once the sort has run
  h->tile_cap = (long long)std::min<unsigned long long>((unsigned long long)cfg->max_blocks * dc.tiles_per_block, (unsigned long long)rec_cap);
  KSG_CUDA(dmalloc(&h->tile_begin, (size_t)h->tile_cap));

  // ---- CUB temp storage: the largest of every call made per frame
  {
    size_t need = 0, t = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, t, h->rec_a, h->rec_b, rec_cap, 0, 64); need = std::max(need, t);
    cub::DeviceRadixSort::SortPairs(nullptr, t, h->pt_key, h->pt_key, h->iota, h->iota, (int)N, 0, 64); need = std::max(need, t);
    cub::DeviceRadixSort::SortPairs(nullptr, t, h->iota, h->iota, h->iota, h->iota, (int)N, 0, 32); need = std::max(need, t);
    cub::DeviceSelect::Flagged(nullptr, t, cub::CountingInputIterator<int>(0), h->flags8, h->pix_list, (int*)nullptr, (int)(2 * N));
    need = std::max(need, t);
    h->cub_temp_bytes = need + 256;
    KSG_CUDA(cudaMalloc(&h->cub_temp, h->cub_temp_bytes));
  }

  // ---- tile-apply launch configuration
  {
    const int V = dc.tile_voxels;
    const size_t stage = dc.head_bytes + (dc.full_stage ? dc.prior_bytes : 0u);
    h->apply_smem = (int)(stage + (size_t)V * 8 + 64);
    h->apply_nch = dc.C <= 32 ? 1 : (dc.C <= 64 ? 2 : (dc.C <= 128 ? 4 : 8));
    h->use_tma = cfg->apply_mode == 0;
#define KSG_ATTR(TMA, NCH) \
    KSG_CUDA(cudaFuncSetAttribute(k_tile_apply<TMA, NCH, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->apply_smem)); \
    KSG_CUDA(cudaFuncSetAttribute(k_tile_apply<TMA, NCH, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->apply_smem))
    KSG_CUDA(cudaFuncSetAttribute(k_tile_apply<true, 1, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->apply_smem));
    KSG_ATTR(true, 1); KSG_ATTR(true, 2); KSG_ATTR(true, 4); KSG_ATTR(true, 8);
    KSG_ATTR(false, 1); KSG_ATTR(false, 2); KSG_ATTR(false, 4); KSG_ATTR(false, 8);
#undef KSG_ATTR
  }
  if (fast) {
    // round-2 frame driver (ksg_fast.cuh)
    h->fast_v2 = true;
    if (const char* e = std::getenv("KSG_FAST_LEGACY")) h->fast_v2 = std::atoi(e) == 0;
    KSG_CUDA(dmalloc(&h->d_fc, 1));
    KSG_CUDA(cudaMemset(h->d_fc, 0, sizeof(FastCounters)));
    KSG_CUDA(cudaMallocHost((void**)&h->h_fc_base, 2 * sizeof(FastCounters)));
    std::memset(h->h_fc_base, 0, 2 * sizeof(FastCounters));
    h->h_fc = h->h_fc_base;
    KSG_CUDA(dmalloc(&h->blk_cnt, N / kCountBlock + 2)); KSG_CUDA(dmalloc(&h->blk_off, N / kCountBlock + 2));
    KSG_CUDA(dmalloc(&h->warp_cnt, N / 32 + 64)); KSG_CUDA(dmalloc(&h->warp_off, N / 32 + 64));
    if (cfg->integration_order_mode == KSG_ORDER_SORTED) KSG_CUDA(dmalloc(&h->seq_of_i, N));
    KSG_CUDA(dmalloc(&h->keys32, (size_t)rec_cap));
    const size_t n_tk = (size_t)h->ht_cap * dc.tiles_per_block;
    KSG_CUDA(dmalloc(&h->tile_cnt, n_tk)); KSG_CUDA(dmalloc(&h->tile_slot, n_tk));
    KSG_CUDA(cudaMemset(h->tile_cnt, 0, sizeof(int) * n_tk));
    KSG_CUDA(dmalloc(&h->tile_list, (size_t)h->tile_cap));
    {
      int per_sm = 0;
      KSG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fast_solve, kSolveThreads, 0));
      int per_sm3 = 0;
      if (const char* e = std::getenv("KSG_SOLVE_THREADS")) { const int t = std::atoi(e); if (t == 256 || t == 512 || t == 1024) h->solve_threads = t; }
      if (const char* e = std::getenv("KSG_GROUP0")) h->group0 = std::max(32, std::atoi(e));
      if (const char* e = std::getenv("KSG_GROUP_MUL")) h->group_mul = std::max(2, std::atoi(e));
      h->solve_smem = (int)(sizeof(int) * kSortPerWarp * (h->solve_threads / 32));
      KSG_CUDA(cudaFuncSetAttribute(k_fast_solve3, cudaFuncAttributeMaxDynamicSharedMemorySize, h->solve_smem));
      KSG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm3, k_fast_solve3, h->solve_threads, (size_t)h->solve_smem));
      if (h->solver == 3) per_sm = per_sm3;
      int coop = 0;
      cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, h->device);
      if (!coop || per_sm <= 0) h->fast_v2 = false;
      h->solve_grid = h->sm_count * std::max(1, per_sm);
      if (const char* e = std::getenv("KSG_SOLVE_CTAS_PER_SM")) h->solve_grid = h->sm_count * std::max(1, std::min(per_sm, std::atoi(e)));
      int khz = 0;
      if (cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, h->device) == cudaSuccess && khz > 0) h->clock_khz = khz;
    }
    {
      const size_t stage = dc.head_bytes + (dc.full_stage ? dc.prior_bytes : 0u);
      h->apply_fast_smem = (int)(stage + (size_t)dc.tile_voxels * 10 + 16 + 2 * sizeof(uint32_t) * kFastKeyCap + 64 + 32 + (size_t)kFastPref * 21);
#define KSG_ATTRF(TMA, NCH) KSG_CUDA(cudaFuncSetAttribute(k_tile_apply_fast<TMA, NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->apply_fast_smem))
      KSG_ATTRF(true, 1); KSG_ATTRF(true, 2); KSG_ATTRF(true, 4); KSG_ATTRF(true, 8);
      KSG_ATTRF(false, 1); KSG_ATTRF(false, 2); KSG_ATTRF(false, 4); KSG_ATTRF(false, 8);
#undef KSG_ATTRF
    }
    KSG_CUDA(dmalloc(&h->d_gridbar, 1));
    int per_sm = 0;
    KSG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_eval_persistent, 256, 0));
    int coop = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, h->device);
    h->eval_grid = h->sm_count * std::max(1, std::min(per_sm, 4));
    // measured on B200 (profiles/README.md): the persistent solver is ~3 % slower than launch-per-sweep (the sweeps, not the
    // launches, dominate), so it is opt-in: KSG_PERSISTENT_EVAL=1
    h->persistent_eval = false;
    if (const char* e = std::getenv("KSG_PERSISTENT_EVAL")) h->persistent_eval = coop != 0 && per_sm > 0 && std::atoi(e) != 0;
  }
  if (const char* e = std::getenv("KSG_SWEEPS_PER_SYNC")) h->sweeps_per_sync = std::max(1, std::min(8, std::atoi(e)));
  if (const char* e = std::getenv("KSG_FIRST_BATCH")) h->first_batch = std::max(1, std::min(8, std::atoi(e)));
  KSG_CUDA(cudaDeviceSynchronize());
  {
    int r2 = reset_map(h, h->own_stream);
    if (r2) { std::string m = h->err; return fail(r2, m.c_str()); }
  }
  *out = h;
  return KSG_OK;
}

void ksg_destroy(ksg_integrator* h) {
  if (!h) return;
  free_all(h);
  delete h;
}

int32_t ksg_set_color_to_label(ksg_integrator* h, const uint8_t* rgb, const uint8_t* labels, int32_t n) {
  if (!h || n < 0 || n > 512 || (n > 0 && (!rgb || !labels))) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  for (int i = 0; i < 1024; ++i) { h->h_luts.c2l_keys[i] = 0xFFFFFFFFu; h->h_luts.c2l_vals[i] = 0; }
  for (int i = 0; i < n; ++i) {
    const uint32_t key = (uint32_t)rgb[3 * i] | ((uint32_t)rgb[3 * i + 1] << 8) | ((uint32_t)rgb[3 * i + 2] << 16);
    uint32_t p = (key * 2654435761u) >> 22;
    while (h->h_luts.c2l_keys[p] != 0xFFFFFFFFu && h->h_luts.c2l_keys[p] != key) p = (p + 1) & 1023;
    h->h_luts.c2l_keys[p] = key;
    h->h_luts.c2l_vals[p] = labels[i];  // later rows overwrite earlier ones (color.cpp:58-59)
  }
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaMemcpy(h->d_luts, &h->h_luts, sizeof(Luts), cudaMemcpyHostToDevice));
  return KSG_OK;
}

int32_t ksg_integrate_points_device(ksg_integrator* h, const float* T, const float* d_xyz, const uint8_t* d_rgba,
                                    const uint8_t* d_labels, int64_t n, int32_t freespace, void* stream, ksg_frame_stats* stats) {
  if (!h || !T || n < 0 || (n > 0 && !d_xyz)) return KSG_ERR_INVALID_ARGUMENT;
  if (h->cfg.integrator_type == KSG_INTEGRATOR_MERGED && d_rgba && d_labels && h->cfg.color_mode == KSG_COLOR_MODE_COLOR)
    return h->fail(KSG_ERR_INVALID_ARGUMENT, "merged, ColorMode::kColor: explicit labels together with point colours (merged.h:82-86 blends the colours, "
                                             "merged.cpp:262-274) are not supported - pass the colours alone (labels by colour) or choose another colour mode");
  InputDesc in; in.d_xyz = d_xyz; in.d_rgba = d_rgba; in.d_labels = d_labels; in.n = n; in.freespace = freespace;
  return integrate(h, in, T, stream ? (cudaStream_t)stream : h->own_stream, stats);
}

int32_t ksg_integrate_depth_device_k64(ksg_integrator* h, const float* T, const float* d_depth, const uint8_t* d_label, int32_t width,
                                       int32_t height, const double* K, void* stream, ksg_frame_stats* stats) {
  if (!h || !T || !K || width <= 0 || height <= 0 || !d_depth || !d_label) return KSG_ERR_INVALID_ARGUMENT;
  InputDesc in; in.d_depth = d_depth; in.d_label_img = d_label; in.width = width; in.height = height;
  in.n = (int64_t)width * height; std::memcpy(in.K, K, sizeof(in.K));
  return integrate(h, in, T, stream ? (cudaStream_t)stream : h->own_stream, stats);
}
int32_t ksg_integrate_depth_device(ksg_integrator* h, const float* T, const float* d_depth, const uint8_t* d_label, int32_t width,
                                   int32_t height, const float* K, void* stream, ksg_frame_stats* stats) {
  if (!K) return KSG_ERR_INVALID_ARGUMENT;
  const double K64[4] = {K[0], K[1], K[2], K[3]};   // exact widening: same results as before for float intrinsics
  return ksg_integrate_depth_device_k64(h, T, d_depth, d_label, width, height, K64, stream, stats);
}

int32_t ksg_integrate_points(ksg_integrator* h, const float* T, const float* xyz, const uint8_t* rgba, const uint8_t* labels,
                             int64_t n, int32_t freespace, ksg_frame_stats* stats) {
  if (!h || !T || n < 0 || (n > 0 && !xyz)) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  if (n > h->cap_points) return fail(KSG_ERR_INVALID_ARGUMENT, "cloud / frame larger than ksg_config.max_points");   // before any staging copy
  if (h->cfg.integrator_type == KSG_INTEGRATOR_MERGED && rgba && labels && h->cfg.color_mode == KSG_COLOR_MODE_COLOR)
    return fail(KSG_ERR_INVALID_ARGUMENT, "merged, ColorMode::kColor: explicit labels together with point colours are not supported (see ksg.h)");
  KSG_CUDA(cudaSetDevice(h->device));
  auto up256 = [](size_t v) { return (v + 255) / 256 * 256; };
  const size_t b_xyz = (size_t)n * 12, b_rgba = rgba ? (size_t)n * 4 : 0, b_lab = labels ? (size_t)n : 0;
  const size_t o_rgba = up256(b_xyz), o_lab = o_rgba + up256(b_rgba);
  const size_t total = o_lab + up256(b_lab) + 256;
  int rc = ensure_input(h, total);
  if (rc) return rc;
  if (n > 0) {
    std::memcpy(h->h_stage, xyz, b_xyz);
    if (rgba) std::memcpy(h->h_stage + o_rgba, rgba, b_rgba);
    if (labels) std::memcpy(h->h_stage + o_lab, labels, b_lab);
    KSG_CUDA(cudaMemcpyAsync(h->d_in, h->h_stage, total, cudaMemcpyHostToDevice, h->own_stream));
  }
  InputDesc in; in.d_xyz = (const float*)h->d_in; in.d_rgba = rgba ? h->d_in + o_rgba : nullptr;
  in.d_labels = labels ? h->d_in + o_lab : nullptr; in.n = n; in.freespace = freespace;
  ksg_frame_stats local;
  return integrate(h, in, T, h->own_stream, stats ? stats : &local);
}

int32_t ksg_integrate_depth_k64(ksg_integrator* h, const float* T, const float* depth, const uint8_t* label, int32_t width,
                                int32_t height, const double* K, ksg_frame_stats* stats) {
  if (!h || !T || !K || width <= 0 || height <= 0 || !depth || !label) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  const size_t P = (size_t)width * height;
  if ((int64_t)P > h->cap_points) return fail(KSG_ERR_INVALID_ARGUMENT, "cloud / frame larger than ksg_config.max_points");   // before any staging copy
  const size_t o_lab = (P * 4 + 255) / 256 * 256;
  const size_t total = o_lab + (P + 255) / 256 * 256;
  int rc = ensure_input(h, total);
  if (rc) return rc;
  if (is_pinned_host(depth) && is_pinned_host(label)) {   // caller's buffers are page-locked: copy straight from them
    KSG_CUDA(cudaMemcpyAsync(h->d_in, depth, P * 4, cudaMemcpyHostToDevice, h->own_stream));
    KSG_CUDA(cudaMemcpyAsync(h->d_in + o_lab, label, P, cudaMemcpyHostToDevice, h->own_stream));
  } else {
    std::memcpy(h->h_stage, depth, P * 4);
    std::memcpy(h->h_stage + o_lab, label, P);
    KSG_CUDA(cudaMemcpyAsync(h->d_in, h->h_stage, total, cudaMemcpyHostToDevice, h->own_stream));
  }
  InputDesc in; in.d_depth = (const float*)h->d_in; in.d_label_img = h->d_in + o_lab; in.width = width; in.height = height;
  in.n = (int64_t)P; std::memcpy(in.K, K, sizeof(in.K));
  ksg_frame_stats local;
  return integrate(h, in, T, h->own_stream, stats ? stats : &local);
}
namespace {
// SemanticLabel2Color::getSemanticLabelFromColor per pixel (color.cpp:69-82, alpha forced to 255 as fast.cpp:157 / merged.cpp:87 do)
__global__ void k_rgb_to_label(const uint8_t* __restrict__ rgb, int n, const Luts* __restrict__ luts, uint8_t* __restrict__ label, uint32_t* __restrict__ color) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t c = (uint32_t)rgb[3 * i] | ((uint32_t)rgb[3 * i + 1] << 8) | ((uint32_t)rgb[3 * i + 2] << 16);
  uint32_t hh = (c * 2654435761u) >> 22;
  uint8_t l = 0;
  for (int p = 0; p < 1024; ++p) {
    const uint32_t k = luts->c2l_keys[hh];
    if (k == c) { l = luts->c2l_vals[hh]; break; }
    if (k == 0xFFFFFFFFu) break;
    hh = (hh + 1) & 1023;
  }
  label[i] = l;
  color[i] = c | 0xFF000000u;
}
}  // namespace

int32_t ksg_integrate_image(ksg_integrator* h, const float* T, const void* depth, int32_t depth_type, const void* semantic, int32_t semantic_type,
                            int32_t width, int32_t height, const double* K, ksg_frame_stats* stats) {
  if (!h || !T || !K || width <= 0 || height <= 0 || !depth || !semantic) return KSG_ERR_INVALID_ARGUMENT;
  if (depth_type != KSG_DEPTH_F32_METRES && depth_type != KSG_DEPTH_U16_MILLIMETRES) return KSG_ERR_INVALID_ARGUMENT;
  if (semantic_type != KSG_SEMANTIC_LABEL_U8 && semantic_type != KSG_SEMANTIC_RGB8) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  const size_t P = (size_t)width * height;
  if ((int64_t)P > h->cap_points) return fail(KSG_ERR_INVALID_ARGUMENT, "cloud / frame larger than ksg_config.max_points");
  auto up = [](size_t v) { return (v + 255) / 256 * 256; };
  const size_t b_depth = P * (depth_type == KSG_DEPTH_U16_MILLIMETRES ? 2 : 4), b_sem = P * (semantic_type == KSG_SEMANTIC_RGB8 ? 3 : 1);
  // device staging: [raw depth | raw semantic | float depth | label | colour]
  const size_t o_sem = up(b_depth), o_f32 = o_sem + up(b_sem), o_lab = o_f32 + up(P * 4), o_col = o_lab + up(P), total = o_col + up(P * 4);
  int rc = ensure_input(h, total);
  if (rc) return rc;
  std::memcpy(h->h_stage, depth, b_depth);
  std::memcpy(h->h_stage + o_sem, semantic, b_sem);
  cudaStream_t s = h->own_stream;
  KSG_CUDA(cudaMemcpyAsync(h->d_in, h->h_stage, o_sem + b_sem, cudaMemcpyHostToDevice, s));
  InputDesc in;
  in.width = width; in.height = height; in.n = (int64_t)P;
  std::memcpy(in.K, K, sizeof(in.K));
  if (depth_type == KSG_DEPTH_U16_MILLIMETRES) {
    ++h->n_launches;
    k_u16_to_f32<<<grid_for((long long)P, 256), 256, 0, s>>>((const uint16_t*)h->d_in, (int)P, (float*)(h->d_in + o_f32));
    in.d_depth = (const float*)(h->d_in + o_f32);
    in.unit_scaling = (double)0.001f;          // double unit_scaling = DepthTraits<uint16_t>::toMeters(1) = 1 * 0.001f
    in.z_scale = 0.001f;
  } else in.d_depth = (const float*)h->d_in;
  if (semantic_type == KSG_SEMANTIC_RGB8) {
    ++h->n_launches;
    k_rgb_to_label<<<grid_for((long long)P, 256), 256, 0, s>>>(h->d_in + o_sem, (int)P, h->d_luts, h->d_in + o_lab, (uint32_t*)(h->d_in + o_col));
    in.d_label_img = h->d_in + o_lab;
    in.d_color_img = (const uint32_t*)(h->d_in + o_col);
  } else in.d_label_img = h->d_in + o_sem;
  ksg_frame_stats local;
  return integrate(h, in, T, s, stats ? stats : &local);
}

int32_t ksg_integrate_depth(ksg_integrator* h, const float* T, const float* depth, const uint8_t* label, int32_t width,
                            int32_t height, const float* K, ksg_frame_stats* stats) {
  if (!K) return KSG_ERR_INVALID_ARGUMENT;
  const double K64[4] = {K[0], K[1], K[2], K[3]};
  return ksg_integrate_depth_k64(h, T, depth, label, width, height, K64, stats);
}

// Pipelined host-buffer entry: the H2D copy of this frame runs on a copy stream into one of two device staging buffers, so it
// overlaps the kernels of the previous frame; the frame's kernels wait for the copy with an event.  Returns without waiting.
int32_t ksg_integrate_depth_async(ksg_integrator* h, const float* T, const float* depth, const uint8_t* label, int32_t width,
                                  int32_t height, const float* K) {
  if (!h || !T || !K || width <= 0 || height <= 0 || !depth || !label) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  const size_t P = (size_t)width * height;
  if ((int64_t)P > h->cap_points) return fail(KSG_ERR_INVALID_ARGUMENT, "cloud / frame larger than ksg_config.max_points");
  const size_t o_lab = (P * 4 + 255) / 256 * 256;
  const size_t total = o_lab + (P + 255) / 256 * 256;
  const int slot = h->in_slot;
  h->in_slot ^= 1;
  if (total > h->in2_bytes[slot]) {
    if (h->in2_used[slot]) KSG_CUDA(cudaEventSynchronize(h->ev_free[slot]));
    if (h->d_in2[slot]) cudaFree(h->d_in2[slot]);
    if (h->h_stage2[slot]) cudaFreeHost(h->h_stage2[slot]);
    h->d_in2[slot] = nullptr; h->h_stage2[slot] = nullptr;
    KSG_CUDA(cudaMalloc((void**)&h->d_in2[slot], total));
    KSG_CUDA(cudaMallocHost((void**)&h->h_stage2[slot], total));
    h->in2_bytes[slot] = total;
  }
  // the slot's previous frame must have consumed the device buffer before it is overwritten
  if (h->in2_used[slot]) KSG_CUDA(cudaStreamWaitEvent(h->copy_stream, h->ev_free[slot], 0));
  if (is_pinned_host(depth) && is_pinned_host(label)) {   // page-locked caller buffers: read asynchronously (keep them unchanged until ksg_wait_frame)
    KSG_CUDA(cudaMemcpyAsync(h->d_in2[slot], depth, P * 4, cudaMemcpyHostToDevice, h->copy_stream));
    KSG_CUDA(cudaMemcpyAsync(h->d_in2[slot] + o_lab, label, P, cudaMemcpyHostToDevice, h->copy_stream));
  } else {
    if (h->in2_used[slot]) KSG_CUDA(cudaEventSynchronize(h->ev_copy[slot]));   // the staging buffer's previous copy has left the host
    std::memcpy(h->h_stage2[slot], depth, P * 4);
    std::memcpy(h->h_stage2[slot] + o_lab, label, P);
    KSG_CUDA(cudaMemcpyAsync(h->d_in2[slot], h->h_stage2[slot], total, cudaMemcpyHostToDevice, h->copy_stream));
  }
  KSG_CUDA(cudaEventRecord(h->ev_copy[slot], h->copy_stream));
  KSG_CUDA(cudaStreamWaitEvent(h->own_stream, h->ev_copy[slot], 0));
  InputDesc in; in.d_depth = (const float*)h->d_in2[slot]; in.d_label_img = h->d_in2[slot] + o_lab; in.width = width; in.height = height;
  in.n = (int64_t)P;
  in.K[0] = K[0]; in.K[1] = K[1]; in.K[2] = K[2]; in.K[3] = K[3];
  const bool deferred = h->cfg.integrator_type == KSG_INTEGRATOR_FAST && h->fast_v2;
  ksg_frame_stats st;
  const int rc = integrate(h, in, T, h->own_stream, deferred ? nullptr : &st);
  KSG_CUDA(cudaEventRecord(h->ev_free[slot], h->own_stream));
  h->in2_used[slot] = true;
  if (!deferred && h->n_stash < 4) h->stash[h->n_stash++] = st;   // drivers that complete inside the call: statistics are ready
  return rc;
}

// Completes the oldest frame submitted with ksg_integrate_depth_async and returns its statistics.
int32_t ksg_wait_frame(ksg_integrator* h, ksg_frame_stats* stats) {
  if (!h) return KSG_ERR_INVALID_ARGUMENT;
  cudaSetDevice(h->device);
  if (h->n_stash > 0) {
    if (stats) *stats = h->stash[0];
    for (int i = 1; i < h->n_stash; ++i) h->stash[i - 1] = h->stash[i];
    --h->n_stash;
    if (h->deferred_status) return h->fail(h->deferred_status, err_text(h->deferred_status));
    return KSG_OK;
  }
  if (h->n_pend > 0) return finish_oldest(h, stats);
  if (stats) fill_stats(h, stats);
  return h->deferred_status ? h->fail(h->deferred_status, err_text(h->deferred_status)) : KSG_OK;
}

int32_t ksg_set_update_log(ksg_integrator* h, int64_t capacity_voxels) {
  if (!h || capacity_voxels < 0 || capacity_voxels > (1ll << 30)) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaDeviceSynchronize());
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  if (h->d_log_head) cudaFree(h->d_log_head);
  if (h->d_log_prior) cudaFree(h->d_log_prior);
  if (h->h_log_head) cudaFreeHost(h->h_log_head);
  if (h->h_log_prior) cudaFreeHost(h->h_log_prior);
  h->d_log_head = nullptr; h->d_log_prior = nullptr; h->h_log_head = nullptr; h->h_log_prior = nullptr; h->log_cap = 0;
  if (capacity_voxels == 0) return KSG_OK;
  if (!(h->cfg.integrator_type == KSG_INTEGRATOR_FAST && h->fast_v2 && h->solver == 3))
    return fail(KSG_ERR_INVALID_ARGUMENT, "the update log is kept by the fast integrator's tile kernel only (merged: use ksg_export_blocks_by_index)");
  const size_t n = (size_t)capacity_voxels;
  KSG_CUDA(cudaMalloc((void**)&h->d_log_head, n * sizeof(VoxelUpdate)));
  KSG_CUDA(cudaMalloc((void**)&h->d_log_prior, n * sizeof(float) * h->dc.C));
  KSG_CUDA(cudaMallocHost((void**)&h->h_log_head, n * sizeof(VoxelUpdate)));
  KSG_CUDA(cudaMallocHost((void**)&h->h_log_prior, n * sizeof(float) * h->dc.C));
  h->log_cap = (int)capacity_voxels;
  return KSG_OK;
}

int32_t ksg_fetch_update_log(ksg_integrator* h, int64_t* n_out, const ksg_voxel_update** heads, const float** priors) {
  if (!h || !n_out) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  *n_out = 0;
  if (!h->d_log_head) return fail(KSG_ERR_INVALID_ARGUMENT, "update log is off (ksg_set_update_log)");
  KSG_CUDA(cudaSetDevice(h->device));
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  const int64_t n = h->h_fc ? h->h_fc->log_count : 0;
  if (n > h->log_cap) { *n_out = -1; return fail(KSG_ERR_SCRATCH_FULL, "update log too small for this frame: fall back to ksg_last_updated_blocks / ksg_export_blocks_by_index"); }
  if (n > 0) {
    KSG_CUDA(cudaMemcpyAsync(h->h_log_head, h->d_log_head, (size_t)n * sizeof(VoxelUpdate), cudaMemcpyDeviceToHost, h->own_stream));
    KSG_CUDA(cudaMemcpyAsync(h->h_log_prior, h->d_log_prior, (size_t)n * sizeof(float) * h->dc.C, cudaMemcpyDeviceToHost, h->own_stream));
    KSG_CUDA(cudaStreamSynchronize(h->own_stream));
  }
  *n_out = n;
  if (heads) *heads = reinterpret_cast<const ksg_voxel_update*>(h->h_log_head);
  if (priors) *priors = h->h_log_prior;
  return KSG_OK;
}

int32_t ksg_evaluate_labels(ksg_integrator* h, const ksg_world_object* objects, int32_t n_objects, float max_dist, float band, float checker_size,
                            float checker_margin, int64_t* evaluated, int64_t* correct, int64_t* observed) {
  if (!h || n_objects < 0 || (n_objects > 0 && !objects) || n_objects > 4096) return KSG_ERR_INVALID_ARGUMENT;
  static_assert(sizeof(ksg_world_object) == sizeof(WorldObject), "ksg_world_object layout");
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaDeviceSynchronize());
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  unsigned long long res[3] = {0, 0, 0};
  if (h->num_blocks > 0 && n_objects > 0) {
    WorldObject* d_objs = nullptr;
    unsigned long long* d_out = nullptr;
    KSG_CUDA(cudaMalloc((void**)&d_objs, sizeof(WorldObject) * (size_t)n_objects));
    KSG_CUDA(cudaMalloc((void**)&d_out, sizeof(res)));
    KSG_CUDA(cudaMemcpy(d_objs, objects, sizeof(WorldObject) * (size_t)n_objects, cudaMemcpyHostToDevice));
    KSG_CUDA(cudaMemset(d_out, 0, sizeof(res)));
    ++h->n_launches;
    k_eval_labels<<<h->sm_count * 4, 256, 0, h->own_stream>>>(h->dc, h->map, (int)h->num_blocks, d_objs, n_objects, max_dist, band, checker_size,
                                                              checker_margin, d_out);
    KSG_CUDA(cudaMemcpyAsync(res, d_out, sizeof(res), cudaMemcpyDeviceToHost, h->own_stream));
    KSG_CUDA(cudaStreamSynchronize(h->own_stream));
    cudaFree(d_objs); cudaFree(d_out);
  }
  if (evaluated) *evaluated = (int64_t)res[0];
  if (correct) *correct = (int64_t)res[1];
  if (observed) *observed = (int64_t)res[2];
  return KSG_OK;
}

static bool key_less_zyx(uint64_t a, uint64_t b);

int32_t ksg_extract_mesh(ksg_integrator* h, float min_weight, int64_t vertex_capacity, float* vertices, uint8_t* rgba, uint8_t* labels,
                         int64_t block_capacity, int32_t* block_index, int64_t* block_first_vertex, int64_t* n_vertices, int64_t* n_blocks) {
  if (!h || vertex_capacity < 0 || block_capacity < 0) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaDeviceSynchronize());
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  const int64_t nb = h->num_blocks;
  if (n_blocks) *n_blocks = nb;
  if (n_vertices) *n_vertices = 0;
  if (nb == 0) { if (block_first_vertex && block_capacity >= 0) block_first_vertex[0] = 0; return KSG_OK; }
  if ((block_index || block_first_vertex) && nb > block_capacity) return fail(KSG_ERR_INVALID_ARGUMENT, "mesh: block capacity too small");
  // blocks in (z, y, x) order, as ksg_export_blocks lists them
  std::vector<uint64_t> keys((size_t)nb);
  KSG_CUDA(cudaMemcpy(keys.data(), h->map.slot_key, sizeof(uint64_t) * nb, cudaMemcpyDeviceToHost));
  std::vector<int> order((size_t)nb);
  for (int64_t i = 0; i < nb; ++i) order[i] = (int)i;
  std::sort(order.begin(), order.end(), [&](int a, int b) { return key_less_zyx(keys[a], keys[b]); });
  int* d_slots = nullptr; int* d_count = nullptr; long long* d_first = nullptr;
  float* d_vtx = nullptr; uint32_t* d_rgba = nullptr; uint8_t* d_label = nullptr;
  auto release = [&]() { cudaFree(d_slots); cudaFree(d_count); cudaFree(d_first); cudaFree(d_vtx); cudaFree(d_rgba); cudaFree(d_label); };
#define KSG_MESH(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { release(); return fail(KSG_ERR_CUDA, cudaGetErrorString(e_)); } } while (0)
  KSG_MESH(cudaMalloc((void**)&d_slots, sizeof(int) * nb));
  KSG_MESH(cudaMalloc((void**)&d_count, sizeof(int) * nb));
  KSG_MESH(cudaMalloc((void**)&d_first, sizeof(long long) * nb));
  KSG_MESH(cudaMemcpy(d_slots, order.data(), sizeof(int) * nb, cudaMemcpyHostToDevice));
  cudaStream_t s = h->own_stream;
  const int grid = (int)std::min<int64_t>(nb, (int64_t)h->sm_count * 8);
  MeshBuf none{nullptr, nullptr, nullptr};
  ++h->n_launches;
  k_mesh_blocks<false><<<grid, kMeshThreads, 0, s>>>(h->dc, h->map, d_slots, (int)nb, min_weight, nullptr, d_count, none);
  std::vector<int> count((size_t)nb);
  KSG_MESH(cudaMemcpyAsync(count.data(), d_count, sizeof(int) * nb, cudaMemcpyDeviceToHost, s));
  KSG_MESH(cudaStreamSynchronize(s));
  std::vector<long long> first((size_t)nb + 1);
  first[0] = 0;
  for (int64_t i = 0; i < nb; ++i) first[i + 1] = first[i] + count[i];
  const int64_t total = first[nb];
  if (n_vertices) *n_vertices = total;
  if (block_index)
    for (int64_t i = 0; i < nb; ++i) {
      const I3 b = unpack_key(keys[order[i]]);
      block_index[3 * i] = b.x; block_index[3 * i + 1] = b.y; block_index[3 * i + 2] = b.z;
    }
  if (block_first_vertex) for (int64_t i = 0; i <= nb && i <= block_capacity; ++i) block_first_vertex[i] = first[i];
  if (!vertices && !rgba && !labels) { release(); return KSG_OK; }                 // counting call
  if (total > vertex_capacity) { release(); return fail(KSG_ERR_INVALID_ARGUMENT, "mesh: vertex capacity too small (n_vertices holds the need)"); }
  if (total > 0) {
    KSG_MESH(cudaMalloc((void**)&d_vtx, sizeof(float) * 3 * total));
    KSG_MESH(cudaMalloc((void**)&d_rgba, sizeof(uint32_t) * total));
    KSG_MESH(cudaMalloc((void**)&d_label, (size_t)total));
    KSG_MESH(cudaMemcpyAsync(d_first, first.data(), sizeof(long long) * nb, cudaMemcpyHostToDevice, s));
    MeshBuf mb{d_vtx, d_rgba, d_label};
    ++h->n_launches;
    k_mesh_blocks<true><<<grid, kMeshThreads, 0, s>>>(h->dc, h->map, d_slots, (int)nb, min_weight, d_first, nullptr, mb);
    if (vertices) KSG_MESH(cudaMemcpyAsync(vertices, d_vtx, sizeof(float) * 3 * total, cudaMemcpyDeviceToHost, s));
    if (rgba) KSG_MESH(cudaMemcpyAsync(rgba, d_rgba, sizeof(uint32_t) * total, cudaMemcpyDeviceToHost, s));
    if (labels) KSG_MESH(cudaMemcpyAsync(labels, d_label, (size_t)total, cudaMemcpyDeviceToHost, s));
    KSG_MESH(cudaStreamSynchronize(s));
    KSG_MESH(cudaGetLastError());
  }
#undef KSG_MESH
  release();
  return KSG_OK;
}

int32_t ksg_sync(ksg_integrator* h) {
  if (!h) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaDeviceSynchronize());
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  if (h->deferred_status) return h->fail(h->deferred_status, err_text(h->deferred_status));
  return KSG_OK;
}

int64_t ksg_num_blocks(ksg_integrator* h) {
  if (!h) return 0;
  if (h->n_pend > 0) { cudaSetDevice(h->device); finish_frame(h, nullptr); }
  return h->num_blocks;
}

static bool key_less_zyx(uint64_t a, uint64_t b) { return a < b; }  // packed as z:y:x, biased -> numeric order = (z, y, x)

static int export_slots(ksg_integrator* h, const std::vector<int>& slots, float* tsdf_distance, float* tsdf_weight,
                        uint8_t* tsdf_rgba, uint8_t* sem_label, float* sem_priors, uint8_t* sem_rgba) {
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  const int64_t nb = (int64_t)slots.size();
  if (nb == 0) return KSG_OK;
  const DevCfg& dc = h->dc;
  const size_t VB = (size_t)dc.vps * dc.vps * dc.vps;
  const size_t per_block = VB * (4 + 4 + 4 + 1 + 4 + 4 * (size_t)dc.C) + 64;
  const int64_t batch = std::max<int64_t>(1, std::min<int64_t>(nb, (int64_t)((256ull << 20) / per_block)));
  if (h->exp_slots_cap < batch) {
    if (h->d_exp_slots) cudaFree(h->d_exp_slots);
    h->d_exp_slots = nullptr;
    KSG_CUDA(dmalloc(&h->d_exp_slots, (size_t)batch));
    h->exp_slots_cap = (int)batch;
  }
  const size_t need = (size_t)batch * per_block;
  if (h->d_exp_bytes < need) {
    if (h->d_exp) cudaFree(h->d_exp);
    h->d_exp = nullptr;
    KSG_CUDA(cudaMalloc((void**)&h->d_exp, need));
    h->d_exp_bytes = need;
  }
  for (int64_t b0 = 0; b0 < nb; b0 += batch) {
    const int64_t cnt = std::min(batch, nb - b0);
    KSG_CUDA(cudaMemcpy(h->d_exp_slots, slots.data() + b0, sizeof(int) * cnt, cudaMemcpyHostToDevice));
    uint8_t* p = h->d_exp;
    float* o_dist = (float*)p; p += cnt * VB * 4;
    float* o_wgt = (float*)p; p += cnt * VB * 4;
    uint32_t* o_rgba = (uint32_t*)p; p += cnt * VB * 4;
    uint32_t* o_srgba = (uint32_t*)p; p += cnt * VB * 4;
    float* o_prior = (float*)p; p += cnt * VB * 4 * dc.C;
    uint8_t* o_label = p;
    k_export<<<h->sm_count * 4, 256, 0, h->own_stream>>>(dc, h->map, h->d_exp_slots, (int)cnt, tsdf_distance ? o_dist : nullptr,
                                                         tsdf_weight ? o_wgt : nullptr, tsdf_rgba ? o_rgba : nullptr,
                                                         sem_label ? o_label : nullptr, sem_priors ? o_prior : nullptr,
                                                         sem_rgba ? o_srgba : nullptr);
    KSG_CUDA(cudaStreamSynchronize(h->own_stream));
    if (tsdf_distance) KSG_CUDA(cudaMemcpy(tsdf_distance + b0 * VB, o_dist, cnt * VB * 4, cudaMemcpyDeviceToHost));
    if (tsdf_weight) KSG_CUDA(cudaMemcpy(tsdf_weight + b0 * VB, o_wgt, cnt * VB * 4, cudaMemcpyDeviceToHost));
    if (tsdf_rgba) KSG_CUDA(cudaMemcpy(tsdf_rgba + b0 * VB * 4, o_rgba, cnt * VB * 4, cudaMemcpyDeviceToHost));
    if (sem_rgba) KSG_CUDA(cudaMemcpy(sem_rgba + b0 * VB * 4, o_srgba, cnt * VB * 4, cudaMemcpyDeviceToHost));
    if (sem_label) KSG_CUDA(cudaMemcpy(sem_label + b0 * VB, o_label, cnt * VB, cudaMemcpyDeviceToHost));
    if (sem_priors) KSG_CUDA(cudaMemcpy(sem_priors + b0 * VB * dc.C, o_prior, cnt * VB * 4 * dc.C, cudaMemcpyDeviceToHost));
  }
  return KSG_OK;
}

int32_t ksg_export_blocks(ksg_integrator* h, int64_t capacity_blocks, int32_t* block_index, float* tsdf_distance,
                          float* tsdf_weight, uint8_t* tsdf_rgba, uint8_t* sem_label, float* sem_priors, uint8_t* sem_rgba) {
  if (!h) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaDeviceSynchronize());
  finish_frame(h, nullptr);
  const int64_t nb = h->num_blocks;
  if (nb > capacity_blocks) return fail(KSG_ERR_INVALID_ARGUMENT, "export capacity too small");
  if (nb == 0) return KSG_OK;
  std::vector<uint64_t> keys((size_t)nb);
  KSG_CUDA(cudaMemcpy(keys.data(), h->map.slot_key, sizeof(uint64_t) * nb, cudaMemcpyDeviceToHost));
  std::vector<int> order((size_t)nb);
  for (int64_t i = 0; i < nb; ++i) order[i] = (int)i;
  std::sort(order.begin(), order.end(), [&](int a, int b) { return key_less_zyx(keys[a], keys[b]); });
  if (block_index)
    for (int64_t i = 0; i < nb; ++i) {
      const I3 b = unpack_key(keys[order[i]]);
      block_index[3 * i] = b.x; block_index[3 * i + 1] = b.y; block_index[3 * i + 2] = b.z;
    }
  if (!tsdf_distance && !tsdf_weight && !tsdf_rgba && !sem_label && !sem_priors && !sem_rgba) return KSG_OK;
  return export_slots(h, order, tsdf_distance, tsdf_weight, tsdf_rgba, sem_label, sem_priors, sem_rgba);
}

int32_t ksg_export_blocks_by_index(ksg_integrator* h, int64_t n, const int32_t* block_index, uint8_t* found, float* tsdf_distance,
                                   float* tsdf_weight, uint8_t* tsdf_rgba, uint8_t* sem_label, float* sem_priors, uint8_t* sem_rgba) {
  if (!h || n < 0 || (n > 0 && !block_index)) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  if (n == 0) return KSG_OK;
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaDeviceSynchronize());
  finish_frame(h, nullptr);
  // host copy of the hash table: look the keys up exactly as the device does
  std::vector<uint64_t> keys((size_t)h->ht_cap);
  std::vector<int> slot_of((size_t)h->ht_cap);
  KSG_CUDA(cudaMemcpy(keys.data(), h->map.ht_keys, sizeof(uint64_t) * h->ht_cap, cudaMemcpyDeviceToHost));
  KSG_CUDA(cudaMemcpy(slot_of.data(), h->map.ht_slot, sizeof(int) * h->ht_cap, cudaMemcpyDeviceToHost));
  std::vector<int> slots;
  std::vector<int64_t> where;
  for (int64_t i = 0; i < n; ++i) {
    I3 b; b.x = block_index[3 * i]; b.y = block_index[3 * i + 1]; b.z = block_index[3 * i + 2];
    int slot = -1;
    if (key_in_range(b)) {
      const uint64_t key = pack_key(b);
      uint32_t pos = mix64(key) & h->map.ht_mask;
      for (uint32_t probe = 0; probe <= h->map.ht_mask; ++probe) {
        if (keys[pos] == key) { slot = slot_of[pos]; break; }
        if (keys[pos] == kEmptyKey) break;
        pos = (pos + 1) & h->map.ht_mask;
      }
    }
    if (found) found[i] = slot >= 0 ? 1 : 0;
    if (slot >= 0) { slots.push_back(slot); where.push_back(i); }
  }
  if (slots.empty()) return KSG_OK;
  const size_t VB = (size_t)h->dc.vps * h->dc.vps * h->dc.vps;
  const size_t C = (size_t)h->dc.C;
  const bool dense = (int64_t)slots.size() == n;
  if (dense) return export_slots(h, slots, tsdf_distance, tsdf_weight, tsdf_rgba, sem_label, sem_priors, sem_rgba);
  // sparse hit list: export compactly, then scatter to the callers positions
  const size_t m = slots.size();
  std::vector<float> d(tsdf_distance ? m * VB : 0), w(tsdf_weight ? m * VB : 0), pr(sem_priors ? m * VB * C : 0);
  std::vector<uint8_t> c1(tsdf_rgba ? m * VB * 4 : 0), c2(sem_rgba ? m * VB * 4 : 0), lb(sem_label ? m * VB : 0);
  int rc = export_slots(h, slots, tsdf_distance ? d.data() : nullptr, tsdf_weight ? w.data() : nullptr, tsdf_rgba ? c1.data() : nullptr,
                        sem_label ? lb.data() : nullptr, sem_priors ? pr.data() : nullptr, sem_rgba ? c2.data() : nullptr);
  if (rc) return rc;
  for (size_t k = 0; k < m; ++k) {
    const size_t i = (size_t)where[k];
    if (tsdf_distance) std::memcpy(tsdf_distance + i * VB, d.data() + k * VB, VB * 4);
    if (tsdf_weight) std::memcpy(tsdf_weight + i * VB, w.data() + k * VB, VB * 4);
    if (tsdf_rgba) std::memcpy(tsdf_rgba + i * VB * 4, c1.data() + k * VB * 4, VB * 4);
    if (sem_rgba) std::memcpy(sem_rgba + i * VB * 4, c2.data() + k * VB * 4, VB * 4);
    if (sem_label) std::memcpy(sem_label + i * VB, lb.data() + k * VB, VB);
    if (sem_priors) std::memcpy(sem_priors + i * VB * C, pr.data() + k * VB * C, VB * C * 4);
  }
  return KSG_OK;
}

int32_t ksg_import_blocks(ksg_integrator* h, int64_t n, const int32_t* block_index, const float* tsdf_distance, const float* tsdf_weight,
                          const uint8_t* tsdf_rgba, const uint8_t* sem_label, const float* sem_priors, const uint8_t* sem_rgba) {
  if (!h || n < 0 || (n > 0 && !block_index)) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  if (h->deferred_status) return h->fail(h->deferred_status, err_text(h->deferred_status));
  if (n == 0) return KSG_OK;
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaDeviceSynchronize());
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  const DevCfg& dc = h->dc;
  // host mirror of the block hash: look up / insert exactly as the device does (linear probing from mix64(key))
  std::vector<uint64_t> keys((size_t)h->ht_cap);
  std::vector<int> slot_of((size_t)h->ht_cap);
  KSG_CUDA(cudaMemcpy(keys.data(), h->map.ht_keys, sizeof(uint64_t) * h->ht_cap, cudaMemcpyDeviceToHost));
  KSG_CUDA(cudaMemcpy(slot_of.data(), h->map.ht_slot, sizeof(int) * h->ht_cap, cudaMemcpyDeviceToHost));
  std::vector<int> slots((size_t)n);
  std::vector<uint8_t> fresh((size_t)n, 0);
  std::vector<uint64_t> new_keys;
  int64_t nb = h->num_blocks;
  for (int64_t i = 0; i < n; ++i) {
    I3 b; b.x = block_index[3 * i]; b.y = block_index[3 * i + 1]; b.z = block_index[3 * i + 2];
    if (!key_in_range(b)) return fail(KSG_ERR_INDEX_RANGE, err_text(5));
    const uint64_t key = pack_key(b);
    uint32_t pos = mix64(key) & h->map.ht_mask;
    for (uint32_t probe = 0;; ++probe) {
      if (probe > h->map.ht_mask) return fail(KSG_ERR_POOL_FULL, err_text(3));
      if (keys[pos] == key) { slots[i] = slot_of[pos]; break; }
      if (keys[pos] == kEmptyKey) {
        if (nb >= h->map.max_blocks) return fail(KSG_ERR_POOL_FULL, err_text(3));
        keys[pos] = key; slot_of[pos] = (int)nb; slots[i] = (int)nb; fresh[i] = 1; new_keys.push_back(key); ++nb;
        break;
      }
      pos = (pos + 1) & h->map.ht_mask;
    }
  }
  if (!new_keys.empty()) {
    KSG_CUDA(cudaMemcpy(h->map.ht_keys, keys.data(), sizeof(uint64_t) * h->ht_cap, cudaMemcpyHostToDevice));
    KSG_CUDA(cudaMemcpy(h->map.ht_slot, slot_of.data(), sizeof(int) * h->ht_cap, cudaMemcpyHostToDevice));
    KSG_CUDA(cudaMemcpy(h->map.slot_key + h->num_blocks, new_keys.data(), sizeof(uint64_t) * new_keys.size(), cudaMemcpyHostToDevice));
    const int pc = (int)nb;
    KSG_CUDA(cudaMemcpy(&h->d_cnt->pool_count, &pc, sizeof(int), cudaMemcpyHostToDevice));
    h->num_blocks = nb;
  }
  const size_t VB = (size_t)dc.vps * dc.vps * dc.vps;
  const size_t per_block = VB * (4 + 4 + 4 + 1 + 4 + 4 * (size_t)dc.C) + 64;
  const int64_t batch = std::max<int64_t>(1, std::min<int64_t>(n, (int64_t)((256ull << 20) / per_block)));
  if (h->exp_slots_cap < batch) {
    if (h->d_exp_slots) cudaFree(h->d_exp_slots);
    h->d_exp_slots = nullptr;
    KSG_CUDA(dmalloc(&h->d_exp_slots, (size_t)batch));
    h->exp_slots_cap = (int)batch;
  }
  const size_t need = (size_t)batch * per_block + (size_t)batch;
  if (h->d_exp_bytes < need) {
    if (h->d_exp) cudaFree(h->d_exp);
    h->d_exp = nullptr;
    KSG_CUDA(cudaMalloc((void**)&h->d_exp, need));
    h->d_exp_bytes = need;
  }
  for (int64_t b0 = 0; b0 < n; b0 += batch) {
    const int64_t cnt = std::min(batch, n - b0);
    KSG_CUDA(cudaMemcpy(h->d_exp_slots, slots.data() + b0, sizeof(int) * cnt, cudaMemcpyHostToDevice));
    uint8_t* p = h->d_exp;
    float* i_dist = (float*)p; p += cnt * VB * 4;
    float* i_wgt = (float*)p; p += cnt * VB * 4;
    uint32_t* i_rgba = (uint32_t*)p; p += cnt * VB * 4;
    uint32_t* i_srgba = (uint32_t*)p; p += cnt * VB * 4;
    float* i_prior = (float*)p; p += cnt * VB * 4 * dc.C;
    uint8_t* i_label = p; p += cnt * VB;
    uint8_t* d_fresh = p;
    if (tsdf_distance) KSG_CUDA(cudaMemcpy(i_dist, tsdf_distance + b0 * VB, cnt * VB * 4, cudaMemcpyHostToDevice));
    if (tsdf_weight) KSG_CUDA(cudaMemcpy(i_wgt, tsdf_weight + b0 * VB, cnt * VB * 4, cudaMemcpyHostToDevice));
    if (tsdf_rgba) KSG_CUDA(cudaMemcpy(i_rgba, tsdf_rgba + b0 * VB * 4, cnt * VB * 4, cudaMemcpyHostToDevice));
    if (sem_rgba) KSG_CUDA(cudaMemcpy(i_srgba, sem_rgba + b0 * VB * 4, cnt * VB * 4, cudaMemcpyHostToDevice));
    if (sem_label) KSG_CUDA(cudaMemcpy(i_label, sem_label + b0 * VB, cnt * VB, cudaMemcpyHostToDevice));
    if (sem_priors) KSG_CUDA(cudaMemcpy(i_prior, sem_priors + b0 * VB * dc.C, cnt * VB * 4 * dc.C, cudaMemcpyHostToDevice));
    KSG_CUDA(cudaMemcpy(d_fresh, fresh.data() + b0, cnt, cudaMemcpyHostToDevice));
    k_import<<<h->sm_count * 4, 256, 0, h->own_stream>>>(dc, h->map, h->d_exp_slots, d_fresh, (int)cnt, tsdf_distance ? i_dist : nullptr,
                                                         tsdf_weight ? i_wgt : nullptr, tsdf_rgba ? i_rgba : nullptr,
                                                         sem_label ? i_label : nullptr, sem_priors ? i_prior : nullptr,
                                                         sem_rgba ? i_srgba : nullptr);
    KSG_CUDA(cudaStreamSynchronize(h->own_stream));
  }
  return KSG_OK;
}

int32_t ksg_device_map_view(ksg_integrator* h, int64_t* n_blocks, int64_t* block_stride_bytes, void** d_pool, void** d_block_keys) {
  if (!h) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaDeviceSynchronize());
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  if (n_blocks) *n_blocks = h->num_blocks;
  if (block_stride_bytes) *block_stride_bytes = (int64_t)h->dc.block_stride;
  if (d_pool) *d_pool = h->map.pool;
  if (d_block_keys) *d_block_keys = h->map.slot_key;
  return KSG_OK;
}

int32_t ksg_copy_map_device(ksg_integrator* h, void* d_dst_pool, void* d_dst_keys, void* stream) {
  if (!h || !d_dst_pool || !d_dst_keys) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  cudaStream_t s = stream ? (cudaStream_t)stream : h->own_stream;
  if (h->num_blocks > 0) {
    KSG_CUDA(cudaMemcpyAsync(d_dst_pool, h->map.pool, (size_t)h->num_blocks * (size_t)h->dc.block_stride, cudaMemcpyDeviceToDevice, s));
    KSG_CUDA(cudaMemcpyAsync(d_dst_keys, h->map.slot_key, (size_t)h->num_blocks * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
  }
  return KSG_OK;
}

int32_t ksg_merge_blocks_device(ksg_integrator* h, int64_t n_blocks, const void* d_block_keys, const void* d_pool_src, void* stream) {
  if (!h || n_blocks < 0 || (n_blocks > 0 && (!d_block_keys || !d_pool_src))) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  if (h->deferred_status) return h->fail(h->deferred_status, err_text(h->deferred_status));
  if (n_blocks == 0) return KSG_OK;
  KSG_CUDA(cudaSetDevice(h->device));
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  cudaStream_t s = stream ? (cudaStream_t)stream : h->own_stream;
  if (h->exp_slots_cap < n_blocks) {
    KSG_CUDA(cudaStreamSynchronize(s));
    if (h->d_exp_slots) cudaFree(h->d_exp_slots);
    h->d_exp_slots = nullptr;
    KSG_CUDA(dmalloc(&h->d_exp_slots, (size_t)n_blocks));
    h->exp_slots_cap = (int)n_blocks;
  }
  h->frame_stamp += 1;
  h->n_launches += 5;
  k_frame_reset<<<1, 1, 0, s>>>(h->d_cnt, 0);
  k_merge_insert<<<grid_for(n_blocks, 256), 256, 0, s>>>(h->d_cnt, h->map, (const uint64_t*)d_block_keys, (int)n_blocks, h->d_exp_slots, h->frame_stamp);
  k_block_init<<<h->sm_count * 4, 256, 0, s>>>(h->dc, h->d_cnt, h->map);
  k_frame_finish<<<1, 1, 0, s>>>(h->d_cnt, h->map);
  k_merge_tiles<<<h->sm_count * 8, 256, 0, s>>>(h->dc, h->d_cnt, h->map, h->d_luts, h->d_exp_slots, (const uint8_t*)d_pool_src, (int)n_blocks);
  KSG_CUDA(cudaGetLastError());
  int rc = fetch_counters(h, s);
  if (rc) return rc;
  h->num_blocks = h->h_cnt->pool_count;
  h->last_blocks_touched = h->h_cnt->n_blocks_touched;
  const int dev_err = h->h_cnt->err;
  if (dev_err) { h->deferred_status = dev_err; return fail(dev_err, err_text(dev_err)); }
  return KSG_OK;
}

int32_t ksg_copy_update_log_device(ksg_integrator* h, int64_t* n_out, void* d_dst_updates, void* d_dst_priors, int64_t capacity, void* stream) {
  if (!h || !n_out) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  *n_out = 0;
  if (!h->d_log_head) return fail(KSG_ERR_INVALID_ARGUMENT, "update log is off (ksg_set_update_log)");
  KSG_CUDA(cudaSetDevice(h->device));
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  const int64_t n = h->h_fc ? h->h_fc->log_count : 0;
  if (n > h->log_cap) { *n_out = -1; return fail(KSG_ERR_SCRATCH_FULL, "update log too small for this frame"); }
  *n_out = n;
  if (!d_dst_updates && !d_dst_priors) return KSG_OK;                 // size query
  if (n > capacity) return fail(KSG_ERR_INVALID_ARGUMENT, "update log copy: capacity too small");
  cudaStream_t s = stream ? (cudaStream_t)stream : h->own_stream;
  if (n > 0) {
    if (d_dst_updates) KSG_CUDA(cudaMemcpyAsync(d_dst_updates, h->d_log_head, (size_t)n * sizeof(VoxelUpdate), cudaMemcpyDeviceToDevice, s));
    if (d_dst_priors) KSG_CUDA(cudaMemcpyAsync(d_dst_priors, h->d_log_prior, (size_t)n * sizeof(float) * h->dc.C, cudaMemcpyDeviceToDevice, s));
  }
  return KSG_OK;
}

int32_t ksg_merge_voxels_device(ksg_integrator* h, int32_t n_deltas, const int64_t* counts, int64_t stride, const void* d_updates, const void* d_priors,
                                void* stream) {
  if (!h || n_deltas < 0 || n_deltas > 16 || stride < 0 || (n_deltas > 0 && (!counts || !d_updates || !d_priors))) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  if (h->deferred_status) return h->fail(h->deferred_status, err_text(h->deferred_status));
  MergeCounts mc{};
  int64_t any = 0;
  for (int g = 0; g < n_deltas; ++g) {
    if (counts[g] < 0 || counts[g] > stride || counts[g] > 0x7fffffff) return KSG_ERR_INVALID_ARGUMENT;
    mc.n[g] = (int)counts[g];
    any += counts[g];
  }
  if (any == 0) return KSG_OK;
  KSG_CUDA(cudaSetDevice(h->device));
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  cudaStream_t s = stream ? (cudaStream_t)stream : h->own_stream;
  const int64_t total = (int64_t)n_deltas * stride;
  if (total > 0x7fffffff) return fail(KSG_ERR_INVALID_ARGUMENT, "merge: n_deltas * stride_entries exceeds 2^31 - 1");
  if (h->exp_slots_cap < total) {
    KSG_CUDA(cudaStreamSynchronize(s));
    if (h->d_exp_slots) cudaFree(h->d_exp_slots);
    h->d_exp_slots = nullptr;
    KSG_CUDA(dmalloc(&h->d_exp_slots, (size_t)total));
    h->exp_slots_cap = (int)total;
  }
  h->frame_stamp += 1;
  h->n_launches += 4 + n_deltas;
  const VoxelUpdate* upd = (const VoxelUpdate*)d_updates;
  const float* pri = (const float*)d_priors;
  k_frame_reset<<<1, 1, 0, s>>>(h->d_cnt, 0);
  k_mergev_insert<<<grid_for(total, 256), 256, 0, s>>>(h->d_cnt, h->map, upd, mc, n_deltas, (long long)stride, h->d_exp_slots, h->frame_stamp);
  k_block_init<<<h->sm_count * 4, 256, 0, s>>>(h->dc, h->d_cnt, h->map);
  k_frame_finish<<<1, 1, 0, s>>>(h->d_cnt, h->map);
  for (int g = 0; g < n_deltas; ++g) {      // frame order: a voxel that several deltas touched is merged delta by delta
    if (mc.n[g] == 0) continue;
    const int grid = (int)std::min<int64_t>((int64_t)h->sm_count * 16, (mc.n[g] + 7) / 8);
    k_mergev_apply<<<std::max(1, grid), 256, 0, s>>>(h->dc, h->map, h->d_luts, upd + (size_t)g * stride, pri + (size_t)g * stride * h->dc.C,
                                                    h->d_exp_slots + (size_t)g * stride, mc.n[g]);
  }
  KSG_CUDA(cudaGetLastError());
  int rc = fetch_counters(h, s);
  if (rc) return rc;
  h->num_blocks = h->h_cnt->pool_count;
  h->last_blocks_touched = h->h_cnt->n_blocks_touched;
  const int dev_err = h->h_cnt->err;
  if (dev_err) { h->deferred_status = dev_err; return fail(dev_err, err_text(dev_err)); }
  return KSG_OK;
}

int64_t ksg_last_updated_blocks(ksg_integrator* h, int64_t capacity_blocks, int32_t* block_index) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  if (h->n_pend > 0) finish_frame(h, nullptr);
  const int64_t n = h->last_blocks_touched;
  if (!block_index || capacity_blocks < n || n == 0) return n;
  cudaDeviceSynchronize();
  std::vector<int> pos((size_t)n);
  if (cudaMemcpy(pos.data(), h->map.touched_list, sizeof(int) * n, cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
  std::vector<uint64_t> all((size_t)h->ht_cap);
  if (cudaMemcpy(all.data(), h->map.ht_keys, sizeof(uint64_t) * h->ht_cap, cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
  std::vector<uint64_t> keys((size_t)n);
  for (int64_t i = 0; i < n; ++i) keys[i] = all[pos[i]];
  std::sort(keys.begin(), keys.end());
  for (int64_t i = 0; i < n; ++i) {
    const I3 b = unpack_key(keys[i]);
    block_index[3 * i] = b.x; block_index[3 * i + 1] = b.y; block_index[3 * i + 2] = b.z;
  }
  return n;
}

int64_t ksg_unordered_map_schedule(int64_t n, int64_t* bucket_count_after_insert) {
  if (n < 0 || (n > 0 && !bucket_count_after_insert)) return -1;
  std::unordered_map<uint64_t, char> probe;
  for (int64_t i = 0; i < n; ++i) {
    probe.emplace((uint64_t)i, 0);
    bucket_count_after_insert[i] = (int64_t)probe.bucket_count();
  }
  return n;
}

int32_t ksg_owner_mask(int32_t voxels_per_side, int32_t shard_rank, int32_t shard_count, int64_t n, const int32_t* block_index,
                       uint8_t* mask) {
  const int vps = voxels_per_side;
  if (vps <= 0 || (vps & (vps - 1)) || n < 0 || (n > 0 && (!block_index || !mask))) return KSG_ERR_INVALID_ARGUMENT;
  const int count = shard_count > 1 ? shard_count : 1;
  if (shard_rank < 0 || shard_rank >= count) return KSG_ERR_INVALID_ARGUMENT;
  const int T = std::min(vps, kTileSideMax), tps = vps / T;
  const size_t V = (size_t)vps * vps * vps;
  for (int64_t b = 0; b < n; ++b) {
    I3 bi; bi.x = block_index[3 * b]; bi.y = block_index[3 * b + 1]; bi.z = block_index[3 * b + 2];
    const uint64_t key = pack_key(bi);
    for (int z = 0; z < vps; ++z)
      for (int y = 0; y < vps; ++y)
        for (int x = 0; x < vps; ++x) {
          const int tile = (x / T) + tps * ((y / T) + tps * (z / T));
          mask[b * V + (size_t)x + (size_t)vps * ((size_t)y + (size_t)vps * z)] = tile_owner(key, tile, count) == shard_rank ? 1 : 0;
        }
  }
  return KSG_OK;
}

int32_t ksg_set_profiling(ksg_integrator* h, int32_t enable) {
  if (!h) return KSG_ERR_INVALID_ARGUMENT;
  cudaSetDevice(h->device);
  if (enable && !h->ev[0]) for (auto& e : h->ev) cudaEventCreate(&e);
  if (enable && h->d_fc && !h->d_prof) {
    if (cudaMalloc(&h->d_prof, sizeof(long long) * kProfSlots) != cudaSuccess) { h->d_prof = nullptr; return KSG_ERR_CUDA; }
    cudaMemset(h->d_prof, 0, sizeof(long long) * kProfSlots);
  }
  h->profiling = enable != 0;
  for (double& m : h->phase_ms) m = 0.0;
  h->prof_frames = 0; h->n_launches = 0; h->n_libcalls = 0;
  return KSG_OK;
}
int32_t ksg_get_profile(ksg_integrator* h, double* phase_ms, int64_t* frames, int64_t* kernel_launches, int64_t* library_calls) {
  if (!h) return KSG_ERR_INVALID_ARGUMENT;
  if (phase_ms) for (int p = 0; p < KSG_NUM_PHASES; ++p) phase_ms[p] = h->phase_ms[p];
  if (frames) *frames = h->prof_frames;
  if (kernel_launches) *kernel_launches = h->n_launches;
  if (library_calls) *library_calls = h->n_libcalls;
  return KSG_OK;
}

namespace {
__global__ void k_chain_debug(const float* __restrict__ terms, long long n, float s0, float* __restrict__ out) {
  const float s = chain_sum_warp(s0, terms, n);
  if ((threadIdx.x & 31) == 0) *out = s;
}
}  // namespace

int32_t ksg_debug_chain_sum(const float* terms, int64_t n, float s0, float* result) {
  if (n < 0 || (n > 0 && !terms) || !result || !(s0 < 0.0f)) return KSG_ERR_INVALID_ARGUMENT;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return KSG_ERR_NO_DEVICE; }
  float *d_terms = nullptr, *d_out = nullptr;
  int32_t rc = KSG_ERR_CUDA;
  if (cudaMalloc((void**)&d_terms, sizeof(float) * (size_t)std::max<int64_t>(n, 1)) == cudaSuccess &&
      cudaMalloc((void**)&d_out, sizeof(float)) == cudaSuccess &&
      (n == 0 || cudaMemcpy(d_terms, terms, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice) == cudaSuccess)) {
    k_chain_debug<<<1, 32>>>(d_terms, (long long)n, s0, d_out);
    if (cudaMemcpy(result, d_out, sizeof(float), cudaMemcpyDeviceToHost) == cudaSuccess) rc = KSG_OK;
  }
  if (d_terms) cudaFree(d_terms);
  if (d_out) cudaFree(d_out);
  return rc;
}

int64_t ksg_debug_tile_times(ksg_integrator* h, int32_t enable, int64_t capacity, int64_t* records_and_cycles) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  if (enable && !h->tile_debug) {
    if (cudaMalloc((void**)&h->tile_debug, sizeof(long long) * 2 * (size_t)h->tile_cap) != cudaSuccess) { h->tile_debug = nullptr; return 0; }
  }
  const int64_t n = std::min<int64_t>(h->h_cnt->n_tiles, h->tile_cap);
  if (h->tile_debug && records_and_cycles && capacity >= n && n > 0)
    cudaMemcpy(records_and_cycles, h->tile_debug, sizeof(long long) * 2 * n, cudaMemcpyDeviceToHost);
  if (!enable && h->tile_debug) { cudaFree(h->tile_debug); h->tile_debug = nullptr; }
  return n;
}

int64_t ksg_debug_fast_timeline(ksg_integrator* h, int64_t* out64, int64_t* sweeps, double* clock_khz) {
  if (!h || !out64 || !h->h_fc) return 0;
  cudaSetDevice(h->device);
  if (h->n_pend > 0) finish_frame(h, nullptr);
  for (int i = 0; i < kTimelineSlots; ++i) out64[i] = (int64_t)h->h_fc->timeline[i];
  for (int i = 0; i < 16; ++i) out64[kTimelineSlots + i] = (int64_t)h->h_fc->dbg[i];
  long long prof[kProfSlots] = {};
  if (h->d_prof) cudaMemcpy(prof, h->d_prof, sizeof(prof), cudaMemcpyDeviceToHost);
  for (int i = 0; i < kProfSlots; ++i) out64[kTimelineSlots + 16 + i] = (int64_t)prof[i];
  if (sweeps) *sweeps = h->h_fc->sweeps_last;
  if (clock_khz) *clock_khz = h->clock_khz;
  return kTimelineSlots + 16 + kProfSlots;
}

int32_t ksg_clear_map(ksg_integrator* h) {
  if (!h) return KSG_ERR_INVALID_ARGUMENT;
  auto fail = [&](int c, const char* m) { return h->fail(c, m); };
  KSG_CUDA(cudaSetDevice(h->device));
  KSG_CUDA(cudaDeviceSynchronize());
  { const int rcp = finish_frame(h, nullptr); if (rcp) return rcp; }
  cudaStream_t s = h->own_stream;
  KSG_CUDA(cudaMemsetAsync(h->map.ht_keys, 0xFF, sizeof(uint64_t) * h->ht_cap, s));
  KSG_CUDA(cudaMemsetAsync(h->map.ht_slot, 0xFF, sizeof(int) * h->ht_cap, s));
  KSG_CUDA(cudaMemsetAsync(h->map.touched_stamp, 0, sizeof(int) * h->ht_cap, s));
  if (h->tile_cnt) KSG_CUDA(cudaMemsetAsync(h->tile_cnt, 0, sizeof(int) * (size_t)h->ht_cap * h->dc.tiles_per_block, s));
  // the block pool restarts at slot 0; everything else in the counter block is per frame (rewritten by the next frame's first kernel)
  // or belongs to the integrator (sweep ids of the observed-set solver, which the slot stamps refer to) and stays
  KSG_CUDA(cudaMemsetAsync(&h->d_cnt->pool_count, 0, sizeof(int), s));
  KSG_CUDA(cudaMemsetAsync(&h->d_cnt->n_blocks_touched, 0, sizeof(int), s));
  KSG_CUDA(cudaMemsetAsync(&h->d_cnt->n_new_blocks, 0, sizeof(int), s));
  h->num_blocks = 0;
  h->last_blocks_touched = 0;
  KSG_CUDA(cudaStreamSynchronize(s));
  return KSG_OK;
}

int32_t ksg_reset(ksg_integrator* h) {
  if (!h) return KSG_ERR_INVALID_ARGUMENT;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  h->n_pend = 0;
  return reset_map(h, h->own_stream);
}

}  // extern "C"
