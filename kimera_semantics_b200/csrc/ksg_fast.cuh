// ksg_fast.cuh — the `fast` integrator's frame without a host in the loop (round 2).
//
// Round 1 drove a 640x480 / 5 cm frame with ~34 launches + ~40 CUB launches and 3-4 blocking counter read-backs (the
// observed-set solver is data dependent).  Here the frame is FIVE launches and no read-back:
//
//   k_fast_count      depth image, 128-bit loads: finite pixels per 1024-pixel block; the last block to finish scans the
//                     block counts (ticket) and resets the frame counters                      (depth entry only)
//   k_fast_classify   image order, 4 pixels / thread (float4 depth + uchar4 label): back-projection, validity, dynamic
//                     labels, T_G_C * p, start cell; the sequence position (voxblox ThreadSafeIndex, A.3) comes from the
//                     inverse of the mixed permutation; start-set visits are pushed with atomics       (fast.cpp:75-92)
//   k_fast_start_eval start_voxel_approx_set_ decision per point + table commit by the slot's first visitor; per-warp counts
//                     of cast points, scanned by the last block                                              (fast.cpp:90)
//   k_fast_solve      ONE persistent cooperative kernel, grid barriers between its phases: compaction of the cast rays,
//                     ray set-up, the observed-set fixpoint sweeps to convergence (device-side test), table commit,
//                     ray emit, and the distribution of the update records to per-tile segments (counting sort by tile:
//                     count, allocate, scatter) + new-block construction                                (fast.cpp:110-141)
//   k_tile_apply_fast one CTA per touched 8^3 tile: TMA-staged tile, the tile's records sorted by (voxel, ray rank) in
//                     shared memory (the reference's per-voxel update order), TSDF + semantic update, TMA write-back
//
// Exactness arguments are those of ksg_kernels.cuh (same device functions for the sets and the update).
#pragma once
#include "ksg_kernels.cuh"

namespace ksg {

static constexpr int kCountBlock = 1024;      // pixels per block of k_fast_count / k_fast_classify (256 threads x 4)
static constexpr int kEvalBlock = 512;        // sequence positions per block of k_fast_start_eval
static constexpr int kSolveThreads = 1024;     // one CTA per SM: a grid barrier is 148 arrivals
static constexpr int kFastKeyCap = 4096;      // update records of one tile sorted in shared memory (more: sorted in place in global memory)
static constexpr int kFastPref = 1024;        // ... and whose per-record operands (point, label, colour) are prefetched into shared memory
static constexpr int kTimelineSlots = 64;
// profiling-only solver counters (FastFrame::prof, not part of FastCounters, which is copied back every frame):
//   [0] overflow entries of the frame, [1] largest slot count, [2] longest overflow chain walked by an evaluation,
//   [4 + 2 i] rays of sweep i found clean by the dirty check alone, [5 + 2 i] rays of sweep i evaluated (i < kProfSweeps)
static constexpr int kProfSlots = 32;
static constexpr int kProfSweeps = (kProfSlots - 4) / 2;

struct FastCounters {      // device-resident state of the frame driver (persistent across frames)
  unsigned int ticket_count, ticket_eval;   // "last block done" tickets
  unsigned int gridbar;                      // grid barrier of k_fast_solve
  int sweep_base;                            // id of the last observed-set sweep ever run (sweep ids are monotonic: slot stamps)
  int sweeps_last;                           // sweeps of the last frame
  int tile_cursor;
  int n_tile_list;
  int pool_base;                             // pool_count before this frame's new blocks
  unsigned long long rec_cursor;             // allocation cursor of the per-tile key segments
  int ovf_count;                             // overflow pool cursor (solver 3)
  int n_mixed;                               // start-set slots visited by more than one start cell this frame
  int m_cursor;                              // allocation cursor of their visitor lists
  int log_count;                             // update-log entries written by the frame (may exceed the capacity: then the log is incomplete)
  long long timeline[kTimelineSlots];        // clock64 of block 0 at the phase boundaries of k_fast_solve (profiling)
  long long dbg[16];                         // profiling only: maxima / counts gathered inside the solve kernel (see ksg_debug_fast_timeline)
};

struct TileDesc { uint32_t tk; int n; long long off; };

// update log (eager host-layer sync of the C++ drop-in classes): one entry per voxel the frame updated, its final state
struct VoxelUpdate { int bx, by, bz; uint32_t lin_label; float dist, wgt; uint32_t rgba, srgba; };   // lin_label = linear voxel index | label << 24

// observed-set solver, third formulation (ksg_fast3.cuh)
// Rank groups (ranks [0, n) are final once converged, so the solver can finish a prefix of the rays before it starts the rest; the
// following groups are group_mul x larger each).  Measured (profiles/r02/tuning_10.log, fast5): 512 -> 2047 fps, 2048 -> 2207, 8192 -> 2393,
// one group for all rays -> 2494: every extra group costs more grid barriers than it saves work, so the default is ONE group
// (KSG_GROUP0 / KSG_GROUP_MUL keep the mechanism reachable).
static constexpr int kGroup0 = 1 << 30;
struct Cand;
struct OvfEnt;
struct RayRec;
struct Obs3 {
  Cand* cand;              // one 16-byte record per materialised ray step
  long long ext_base, cand_cap;
  int* slot_cnt;           // [2^20] performed-ever candidates of the slot this frame (cleared per frame)
  uint64_t* bkt;           // [2^20][kBktK] entries [performed:1][order:39][value >> 20 : 13]
  int* head;               // [2^20] overflow list head (cleared to -1 per frame)
  OvfEnt* ovf;             // overflow pool (slots with more than kBktK performed-ever candidates)
  int ovf_cap;
  uint64_t* stamp_max;     // [2^20] max over the toggles of the slot of (sweep << 32 | ray)
  uint64_t* stamp_min;     // [2^20] min over the toggles of ((~sweep) << 32 | ray)
  uint32_t* table;         // persistent compact table: value >> 20
};

// everything the fast frame kernels need (passed by value)
struct FastFrame {
  DevCfg cfg;
  Xform T;
  FrameIn in;
  const Luts* luts;
  Counters* cnt;
  FastCounters* fc;
  MapRef map;
  ObsBuf ob;
  StartBuf sb;
  uint64_t set_offset;
  int capacity;              // host upper bound of the point count (pixels or points)
  int n_count_blocks;        // blocks of k_fast_count / k_fast_classify (depth entry)
  int vec_ok;                // depth / label pointers allow 128-bit / 32-bit vector loads
  int frame_stamp;
  int profile;
  long long* prof;           // [kProfSlots] (profiling only)
  const int* seq_of_i;       // "sorted" order mode: sequence position of input index i, else NULL (mixed: closed form)
  int* block_cnt; int* block_off;     // finite pixels per 1024-pixel block
  int* warp_cnt; int* warp_off;       // cast points per 32 sequence positions
  // per sequence position
  float4* pt_pG; uint8_t* pt_label; uint8_t* pt_flags; uint32_t* pt_color; uint64_t* pt_key; uint8_t* cast_flag;
  // per cast ray
  int* cast_seq; float4* ray_param; uint8_t* ray_label; uint8_t* ray_flags; uint32_t* ray_color;
  int* nsteps; int* H; int* L; RayState* ray_state; long long* ext_off; int* eval_sweep;
  // update records
  uint64_t* rec; long long rec_cap;
  uint32_t* keys;            // per-tile segments of (voxel << 23 | ray rank)
  int* tile_cnt;             // [hash capacity * tiles_per_block] records of the tile this frame (returns to 0 by itself)
  int* tile_slot;            // ... index of the tile in tile_list
  TileDesc* tile_list; long long tile_cap;
  // solver 3
  Obs3 o3;
  RayRec* rayrec;
  int* blk_run;              // consecutive-collision count at the start of every evaluation block (index: candidate index / 16)
  int group0, group_mul;     // rank groups of the solver: first group, growth factor
  // update log (NULL: off)
  VoxelUpdate* log_head; float* log_prior; int log_cap;
  // start set, third formulation: per-slot aggregates only (no linked lists)
  int* s_visits;             // [2^20] visitors of the slot this frame (sb.next[seq] = arrival index of the point)
  uint32_t *s_hmin, *s_hmax; // [2^20] smallest / largest (value >> 20) among the visitors: different <=> several cells share the slot
  int* s_base;               // [2^20] start of the slot's visitor list in m_list (slots shared by several cells only)
  int* mixed_list;           // such slots
  int* m_list;               // their visitors (sequence positions), grouped by slot
};

__device__ __forceinline__ int inv_mixed_index(int i, int n) {   // inverse of mixed_index (voxblox MixedThreadSafeIndex, A.3)
  const int groups = n / 1024;
  if (groups * 1024 <= i) return i;
  return (i % 1024) * groups + i / 1024;
}

// exclusive scan of a[0..n) into out[0..n) by ONE block (every thread of the block calls it); returns the total.  a and out are
// 16-byte aligned; every thread owns a contiguous run whose length is a multiple of four (128-bit loads and stores, all independent).
__device__ __forceinline__ int block_scan_array(const int* a, int* out, int n) {
  __shared__ int s_w[32];
  __shared__ int s_total;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nthreads = blockDim.x, nwarps = nthreads >> 5;
  const int per = (((n + nthreads - 1) / nthreads) + 3) & ~3;
  const int i0 = min(n, tid * per), i1 = min(n, i0 + per);
  int local = 0;
  {
    int i = i0;
    for (; i + 4 <= i1; i += 4) { const int4 v = __ldcg((const int4*)(a + i)); local += v.x + v.y + v.z + v.w; }
    for (; i < i1; ++i) local += __ldcg(&a[i]);
  }
  int incl = local;
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) s_w[wid] = incl;
  __syncthreads();
  if (tid == 0) { int t = 0; for (int w = 0; w < nwarps; ++w) { const int v = s_w[w]; s_w[w] = t; t += v; } s_total = t; }
  __syncthreads();
  int run = s_w[wid] + incl - local;
  {
    int i = i0;
    for (; i + 4 <= i1; i += 4) {
      const int4 v = __ldcg((const int4*)(a + i));
      int4 r; r.x = run; r.y = run + v.x; r.z = r.y + v.y; r.w = r.z + v.z;
      *(int4*)(out + i) = r;
      run = r.w + v.w;
    }
    for (; i < i1; ++i) { const int v = __ldcg(&a[i]); out[i] = run; run += v; }
  }
  return s_total;
}

__device__ __forceinline__ void frame_counters_reset(Counters* c, int n_points) {
  c->n_points = n_points; c->n_valid = 0; c->n_cast = 0;
  c->n_new_blocks = 0; c->n_tiles = 0; c->n_blocks_touched = 0; c->tile_cursor = 0; c->n_big_tiles = 0; c->n_small_tiles = 0;
  for (int i = 0; i < 4; ++i) { c->changed[i] = 0; c->n_truncated[i] = 0; c->sum_updates[i] = 0; }
  c->n_records = 0; c->n_skipped = 0; c->n_cand_ext = 0; c->ray_steps = 0;
}

// ---------------------------------------------------------------------------------------------
// k_fast_count: finite pixels per block (depth_map_to_pointcloud.h:259: DepthTraits<float>::valid = isfinite)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_depth4(const float* __restrict__ depth, int p0, int P, int vec_ok, float d[4], int& npx) {
  npx = P - p0; if (npx > 4) npx = 4; if (npx < 0) npx = 0;
  if (npx == 4 && vec_ok) { const float4 v = __ldg((const float4*)(depth + p0)); d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w; }
  else { for (int k = 0; k < 4; ++k) d[k] = (k < npx) ? __ldg(depth + p0 + k) : 0.0f; }
}

__global__ void __launch_bounds__(256) k_fast_count(FastFrame f) {
  __shared__ int s_w[8];
  __shared__ int s_last;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int p0 = blockIdx.x * kCountBlock + tid * 4;
  float d[4]; int npx;
  load_depth4(f.in.depth, p0, f.capacity, f.vec_ok, d, npx);
  int c = 0;
  for (int k = 0; k < 4; ++k) c += (k < npx && isfinite(d[k])) ? 1 : 0;
  for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
  if (lane == 0) s_w[wid] = c;
  __syncthreads();
  if (tid == 0) {
    int t = 0; for (int w = 0; w < 8; ++w) t += s_w[w];
    __stcg(&f.block_cnt[blockIdx.x], t);
    __threadfence();
    s_last = (atomicAdd(&f.fc->ticket_count, 1u) == (unsigned)(f.n_count_blocks - 1));
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const int total = block_scan_array(f.block_cnt, f.block_off, f.n_count_blocks);
  if (tid == 0) { frame_counters_reset(f.cnt, total); f.fc->ticket_count = 0; }
}
// points entry: every point counts
__global__ void k_fast_reset(FastFrame f) { frame_counters_reset(f.cnt, f.capacity); }

// ---------------------------------------------------------------------------------------------
// k_fast_classify: per input point (image order) — fast.cpp:152-158, :75-81, :87-89 — + start-set push
// ---------------------------------------------------------------------------------------------
template <bool PUSH3>
__device__ __forceinline__ void fast_classify_one(const FastFrame& f, int seq, F3 pC, uint8_t label, uint32_t color, bool& valid) {
  const DevCfg& cfg = f.cfg;
  if ((int)label >= cfg.C) { set_err(f.cnt, 1 /*CHECK_LT fast.cpp:134*/); label = 0; }
  const float ray_distance = norm3(pC);                      // isPointValid (A.6)
  valid = true;
  bool clearing = false;
  if (ray_distance < cfg.min_ray) valid = false;
  else if (ray_distance > cfg.max_ray) { if (cfg.allow_clear || f.in.freespace) clearing = true; else valid = false; }
  else clearing = f.in.freespace != 0;
  if (!(ray_distance == ray_distance)) valid = false;
  if (f.luts->dynamic_label[label]) valid = false;           // isSemanticLabelValid (base.h:170-175)
  float w;                                                   // getVoxelWeight (A.6)
  if (cfg.const_weight) w = 1.0f;
  else { const float z = fabsf(pC.z); w = (z > kEps) ? 1.0f / (z * z) : 0.0f; }
  const F3 pG = xform_apply(f.T, pC);
  f.pt_pG[seq] = make_float4(pG.x, pG.y, pG.z, w);
  f.pt_label[seq] = label;
  f.pt_color[seq] = color;
  f.pt_flags[seq] = (valid ? 1 : 0) | (clearing ? 2 : 0);
  uint64_t key = ~0ull;
  if (valid) {
    const F3 sc = mul(pG, cfg.start_inv);
    if (!index_in_range(sc)) set_err(f.cnt, 5);
    const I3 g = grid_index(pG, cfg.start_inv);              // fast.cpp:88-89
    key = (uint64_t)index_hash(g) + f.set_offset;            // ApproxHashSet value = hash + offset_
    const uint32_t slot = (uint32_t)key & kSetMask, hi = (uint32_t)(key >> kSetBits);
    if (PUSH3) {   // aggregates only: no result of these atomics steers the thread, so the four points of a thread overlap
      f.sb.next[seq] = atomicAdd(&f.s_visits[slot], 1);
      atomicMin(&f.sb.smin[slot], seq);
      atomicMax(&f.sb.smax[slot], seq);
      atomicMin(&f.s_hmin[slot], hi);
      atomicMax(&f.s_hmax[slot], hi);
    } else {
      f.sb.next[seq] = atomicExch(&f.sb.head[slot], seq);
      atomicMin(&f.sb.smin[slot], seq);
      atomicMax(&f.sb.smax[slot], seq);
      const uint32_t old = atomicCAS(&f.sb.sval[slot], 0xFFFFFFFFu, hi);
      if (old != 0xFFFFFFFFu && old != hi) f.sb.mixed[slot] = 1;
    }
  }
  f.pt_key[seq] = key;
}

template <bool DEPTH, bool PUSH3>
__global__ void __launch_bounds__(256) k_fast_classify(FastFrame f) {
  __shared__ int s_w[8];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n = f.cnt->n_points;
  int nvalid = 0;
  if (DEPTH) {
    const int p0 = blockIdx.x * kCountBlock + tid * 4;
    float d[4]; int npx;
    load_depth4(f.in.depth, p0, f.capacity, f.vec_ok, d, npx);
    uint8_t lab[4] = {0, 0, 0, 0};
    if (npx == 4 && f.vec_ok) { const uchar4 v = __ldg((const uchar4*)(f.in.label_img + p0)); lab[0] = v.x; lab[1] = v.y; lab[2] = v.z; lab[3] = v.w; }
    else { for (int k = 0; k < npx; ++k) lab[k] = __ldg(f.in.label_img + p0 + k); }
    int c = 0;
    for (int k = 0; k < 4; ++k) c += (k < npx && isfinite(d[k])) ? 1 : 0;
    int incl = c;
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) s_w[wid] = incl;
    __syncthreads();
    int base = f.block_off[blockIdx.x];
    for (int w = 0; w < wid; ++w) base += s_w[w];
    int i = base + incl - c;                                  // index of this thread's first finite pixel among all finite pixels
    for (int k = 0; k < npx; ++k) {
      if (!isfinite(d[k])) continue;
      const int pix = p0 + k;
      const int v = pix / f.in.width, u = pix - v * f.in.width;
      const F3 pC = f3(((float)u - f.in.cx) * d[k] * f.in.constant_x, ((float)v - f.in.cy) * d[k] * f.in.constant_y, d[k] * f.in.z_scale);
      const int seq = f.seq_of_i ? f.seq_of_i[i] : inv_mixed_index(i, n);
      bool valid;
      fast_classify_one<PUSH3>(f, seq, pC, lab[k], f.in.color_img ? f.in.color_img[pix] : f.luts->label_rgba[lab[k]], valid);
      nvalid += valid ? 1 : 0;
      ++i;
    }
  } else {
    const int i = blockIdx.x * blockDim.x + tid;
    if (i < n) {
      const FrameIn& in = f.in;
      const F3 pC = f3(in.xyz[3 * i], in.xyz[3 * i + 1], in.xyz[3 * i + 2]);
      uint32_t color = 0;
      uint8_t label = 0;
      if (in.rgba) color = (uint32_t)in.rgba[4 * i] | ((uint32_t)in.rgba[4 * i + 1] << 8) | ((uint32_t)in.rgba[4 * i + 2] << 16) | ((uint32_t)in.rgba[4 * i + 3] << 24);
      if (in.labels) label = in.labels[i];
      else if (in.rgba) {  // SemanticLabel2Color::getSemanticLabelFromColor (color.cpp:69-82), alpha forced to 255
        const uint32_t rgb = color & 0x00FFFFFFu;
        uint32_t hh = (rgb * 2654435761u) >> 22;
        for (int p = 0; p < 1024; ++p) {
          const uint32_t k = f.luts->c2l_keys[hh];
          if (k == rgb) { label = f.luts->c2l_vals[hh]; break; }
          if (k == 0xFFFFFFFFu) break;
          hh = (hh + 1) & 1023;
        }
      }
      if (!in.rgba) color = f.luts->label_rgba[label];
      const int seq = f.seq_of_i ? f.seq_of_i[i] : inv_mixed_index(i, n);
      bool valid;
      fast_classify_one<PUSH3>(f, seq, pC, label, color, valid);
      nvalid = valid ? 1 : 0;
    }
  }
  for (int o = 16; o > 0; o >>= 1) nvalid += __shfl_down_sync(0xffffffffu, nvalid, o);
  if (lane == 0 && nvalid) atomicAdd(&f.cnt->n_valid, nvalid);
}

// "sorted" order mode (voxblox SortedThreadSafeIndex, A.3): squared norm per input index, image order
__global__ void __launch_bounds__(256) k_fast_sqnorm(FastFrame f, uint32_t* __restrict__ keys) {
  __shared__ int s_w[8];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int p0 = blockIdx.x * kCountBlock + tid * 4;
  float d[4]; int npx;
  load_depth4(f.in.depth, p0, f.capacity, f.vec_ok, d, npx);
  int c = 0;
  for (int k = 0; k < 4; ++k) c += (k < npx && isfinite(d[k])) ? 1 : 0;
  int incl = c;
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) s_w[wid] = incl;
  __syncthreads();
  int base = f.block_off[blockIdx.x];
  for (int w = 0; w < wid; ++w) base += s_w[w];
  int i = base + incl - c;
  for (int k = 0; k < npx; ++k) {
    if (!isfinite(d[k])) continue;
    const int pix = p0 + k;
    const int v = pix / f.in.width, u = pix - v * f.in.width;
    const F3 pC = f3(((float)u - f.in.cx) * d[k] * f.in.constant_x, ((float)v - f.in.cy) * d[k] * f.in.constant_y, d[k] * f.in.z_scale);
    keys[i++] = __float_as_uint(dot3(pC, pC));
  }
}
__global__ void k_fast_sqnorm_points(FastFrame f, uint32_t* __restrict__ keys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= f.capacity) return;
  const F3 pC = f3(f.in.xyz[3 * i], f.in.xyz[3 * i + 1], f.in.xyz[3 * i + 2]);
  keys[i] = __float_as_uint(dot3(pC, pC));
}
__global__ void k_fast_pad_keys(const Counters* cnt, int capacity, uint32_t* __restrict__ keys) {   // positions behind the finite count sort last
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < capacity && i >= cnt->n_points) keys[i] = 0xFFFFFFFFu;
}
__global__ void k_fast_invert_perm(const Counters* cnt, const uint32_t* __restrict__ point_of_seq, int* __restrict__ seq_of_i) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < cnt->n_points) seq_of_i[point_of_seq[s]] = s;
}

// ---------------------------------------------------------------------------------------------
// k_fast_start_eval: start_voxel_approx_set_.replaceHash (fast.cpp:90, A.4) for every point + table commit.
// The set's state is the value of the last visit: a point is cast iff the previous visitor of its slot (sequence order; before
// the first visitor: the persistent table) carried a different value.  Only the slot's FIRST visitor ever reads the table, so
// the same thread also writes the slot's final state (the value of its LAST visitor) — no second kernel.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kEvalBlock) k_fast_start_eval(FastFrame f, int n_eval_blocks) {
  __shared__ int s_last;
  const int seq = blockIdx.x * kEvalBlock + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const StartBuf& sb = f.sb;
  uint8_t cast = 0;
  if (seq < f.cnt->n_points) {
    const uint64_t v = f.pt_key[seq];
    if (v != ~0ull) {
      const uint32_t slot = (uint32_t)v & kSetMask, hi = (uint32_t)(v >> kSetBits);
      const int first = sb.smin[slot];
      if (first == seq) {
        cast = sb.table[slot] != hi;
        ((uint32_t*)sb.table)[slot] = (uint32_t)(f.pt_key[sb.smax[slot]] >> kSetBits);   // state after the frame = last visitor's value
      } else if (sb.mixed[slot]) {
        int best = -1;
        for (int e = sb.head[slot]; e >= 0; e = sb.next[e]) if (e < seq && e > best) best = e;
        cast = f.pt_key[best] != v;           // best >= 0: the first visitor precedes every other one
      }
    }
  }
  if (seq < f.capacity) f.cast_flag[seq] = cast;
  const unsigned m = __ballot_sync(0xffffffffu, cast != 0);
  if (lane == 0) __stcg(&f.warp_cnt[seq >> 5], __popc(m));
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = (atomicAdd(&f.fc->ticket_eval, 1u) == (unsigned)(n_eval_blocks - 1));
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const int n_warps = n_eval_blocks * (kEvalBlock / 32);
  const int total = block_scan_array(f.warp_cnt, f.warp_off, n_warps);
  if (threadIdx.x == 0) { f.cnt->n_cast = total; f.fc->ticket_eval = 0; f.fc->gridbar = 0; }
}

// Third formulation (solver 3): per-slot aggregates instead of linked lists.  Slots visited by ONE start cell (the normal case) are
// decided here as above.  A slot shared by several cells (20-bit aliasing, a few hundred per frame) needs every visitor's predecessor in
// sequence order: its first visitor reserves a list for it; the solve kernel fills, sorts and decides those lists with one warp per slot
// (round 1 let every visitor walk the slot's linked list: the longest list was the critical path of the kernel, 88 us).
__global__ void __launch_bounds__(kEvalBlock) k_fast_start_eval3(FastFrame f) {
  const int seq = blockIdx.x * kEvalBlock + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const StartBuf& sb = f.sb;
  uint8_t cast = 0;
  if (seq < f.cnt->n_points) {
    const uint64_t v = f.pt_key[seq];
    if (v != ~0ull) {
      const uint32_t slot = (uint32_t)v & kSetMask, hi = (uint32_t)(v >> kSetBits);
      if (sb.smin[slot] == seq) {
        cast = sb.table[slot] != hi;
        ((uint32_t*)sb.table)[slot] = (uint32_t)(f.pt_key[sb.smax[slot]] >> kSetBits);   // state after the frame = last visitor's value
        if (f.s_hmin[slot] != f.s_hmax[slot]) {
          f.s_base[slot] = atomicAdd(&f.fc->m_cursor, f.s_visits[slot]);
          f.mixed_list[atomicAdd(&f.fc->n_mixed, 1)] = (int)slot;
        }
      }
    }
  }
  if (seq < f.capacity) f.cast_flag[seq] = cast;
  const unsigned m = __ballot_sync(0xffffffffu, cast != 0);
  if (lane == 0) __stcg(&f.warp_cnt[seq >> 5], __popc(m));
  if (blockIdx.x == 0 && threadIdx.x == 0) f.fc->gridbar = 0;
}

// ascending sort of a[0..n) by one warp (same network as cta_sort_u32 below)
__device__ __forceinline__ void warp_sort_i32(int* a, int n, int lane) {
  int n2 = 1;
  while (n2 < n) n2 <<= 1;
  const int half = n2 >> 1;
  // k and j are powers of two: shifts and masks instead of integer divisions (the sort of a slot with a few hundred visitors is
  // ~360 dependent compare-exchange rounds of one warp, and the divisions were most of each round)
  for (int lk = 1; (1 << lk) <= n2; ++lk) {
    const int k = 1 << lk, lhk = lk - 1;
    for (int t = lane; t < half; t += 32) {
      const int blk = t >> lhk, o = t & ((1 << lhk) - 1);
      const int i = blk * k + o, p = blk * k + (k - 1 - o);
      if (p < n) { const int x = a[i], y = a[p]; if (x > y) { a[i] = y; a[p] = x; } }
    }
    __syncwarp();
    for (int lj = lk - 2; lj >= 0; --lj) {
      const int j = 1 << lj;
      for (int t = lane; t < half; t += 32) {
        const int i = ((t >> lj) << (lj + 1)) + (t & (j - 1)), p = i + j;
        if (p < n) { const int x = a[i], y = a[p]; if (x > y) { a[i] = y; a[p] = x; } }
      }
      __syncwarp();
    }
  }
}

// ---------------------------------------------------------------------------------------------
// k_fast_solve
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void solve_barrier(unsigned int* bar, unsigned int& epoch) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int target = (++epoch) * gridDim.x;
    atomicAdd(bar, 1u);
    while (((volatile unsigned int*)bar)[0] < target) {}
    __threadfence();
  }
  __syncthreads();
}
// Profiling probes of the solve kernel gather per CTA in shared memory and reach global memory once per CTA and phase (prof_flush):
// one same-address global atomic per ray made the profiled frame 1.6x the timed one and moved the phases it measured.
// Slots 0..15: FastCounters::dbg (kDbgAddMask: sums, the others maxima); 16, 17: maxima of prof[1], prof[2]; 18, 19: this sweep's
// prof[4 + 2 i], prof[5 + 2 i].
static constexpr int kDbgShared = 20;
static constexpr unsigned kDbgAddMask = (1u << 4) | (1u << 5) | (1u << 6) | (1u << 7) | (1u << 9);
__shared__ unsigned long long s_dbg[kDbgShared];
__device__ __forceinline__ void dbg_max(const FastFrame& f, int k, long long v) { if (f.profile) atomicMax(&s_dbg[k], (unsigned long long)v); }
__device__ __forceinline__ void dbg_add(const FastFrame& f, int k, long long v) { if (f.profile) atomicAdd(&s_dbg[k], (unsigned long long)v); }
__device__ __forceinline__ void prof_init(const FastFrame& f) {
  if (!f.profile) return;
  if (threadIdx.x < kDbgShared) s_dbg[threadIdx.x] = 0;
  __syncthreads();
}
// every thread of the CTA calls it before a grid barrier; `sweep_idx` is the index of the sweep that just ended (-1: none)
__device__ __forceinline__ void prof_flush(const FastFrame& f, int sweep_idx) {
  if (!f.profile) return;
  __syncthreads();
  const int k = threadIdx.x;
  if (k < kDbgShared) {
    const unsigned long long v = s_dbg[k];
    if (v) {
      if (k < 16) {
        if ((kDbgAddMask >> k) & 1u) atomicAdd((unsigned long long*)&f.fc->dbg[k], v); else atomicMax((unsigned long long*)&f.fc->dbg[k], v);
      } else if (k < 18) atomicMax((unsigned long long*)&f.prof[k - 15], v);
      else if (sweep_idx >= 0 && sweep_idx < kProfSweeps) atomicAdd((unsigned long long*)&f.prof[4 + 2 * sweep_idx + (k - 18)], v);
      s_dbg[k] = 0;
    }
  }
}
__device__ __forceinline__ void timeline_mark(const FastFrame& f, int slot) {
  if (f.profile && blockIdx.x == 0 && threadIdx.x == 0 && slot < kTimelineSlots) f.fc->timeline[slot] = clock64();
}

__device__ __forceinline__ void fast_ray_setup(const FastFrame& f, int r, int n_cast) {
  const DevCfg& cfg = f.cfg;
  int h = 0;
  if (r < n_cast) {
    const int seq = f.cast_seq[r];
    const float4 p = f.pt_pG[seq];
    const uint8_t fl = f.pt_flags[seq];
    f.ray_param[r] = p;
    f.ray_label[r] = f.pt_label[seq];
    f.ray_flags[r] = fl;
    f.ray_color[r] = f.pt_color[seq];
    Dda d;
    raycaster_init(d, f3(f.T.tx, f.T.ty, f.T.tz), f3(p.x, p.y, p.z), (fl & 2) != 0, cfg.carving != 0, cfg.max_ray, cfg.vsi, cfg.tp.trunc,
                   /*cast_from_origin=*/false);
    int n = d.length_in_steps + 1;
    if (!d.in_range || n >= (1 << kOrderStepBits)) { set_err(f.cnt, 5); n = 0; }
    f.nsteps[r] = n;
    h = n < kH0 ? n : kH0;
    const int l0 = h < cfg.maxc ? h : cfg.maxc;   // a ray cannot break before `maxc` consecutive collisions
    for (int s = 0; s < h; ++s) {
      const I3 g = dda_next(d);
      const long long ci = (long long)r * kH0 + s;
      cand_store(f.ob, ci, (uint64_t)index_hash(g) + f.set_offset, ((uint64_t)r << kOrderStepBits) | (uint64_t)s);
      if (s < l0) cand_insert_performed(f.ob, ci);
    }
    RayState st; save_state(st, d); f.ray_state[r] = st;
    f.H[r] = h;
    f.L[r] = l0;
    f.eval_sweep[r] = 0;
  }
  warp_add(&f.cnt->ray_steps, (unsigned long long)h);
}

// After convergence: the last performed visit of every slot becomes the persistent table entry (8 lanes per ray).
__device__ __forceinline__ void fast_obs_commit(const FastFrame& f, int n_cast) {
  constexpr int G = 8;
  const ObsBuf& ob = f.ob;
  const int groups_total = (gridDim.x * blockDim.x) / G;
  const int gl = threadIdx.x % G;
  const int gt = ((((threadIdx.x >> 5) * gridDim.x + blockIdx.x) << 5) | (threadIdx.x & 31));   // CTA-balanced, see k_fast_solve
  for (int r = gt / G; r < n_cast; r += groups_total) {
    const int U = f.L[r];
    for (int s = gl; s < U; s += G) {
      const uint64_t v = __ldcg(&ob.cand_val[cand_index(ob, f.ext_off, r, s)]);
      const uint32_t slot = (uint32_t)v & kSetMask;
      const uint64_t my_order = ((uint64_t)r << kOrderStepBits) | (uint64_t)s;
      const int total = __ldcg(&ob.slot_cnt[slot]);
      const int n = total < kBktK ? total : kBktK;
      const uint64_t* b = ob.bkt + (size_t)slot * kBktK;
      bool later = false;
      for (int j = 0; j < n; ++j) {
        const uint64_t e = __ldcg(&b[j]);
        if ((e & kEntPerf) && ((e >> 13) & ((1ull << kEntOrderBits) - 1)) > my_order) later = true;
      }
      int guard = total - kBktK + 8;
      if (total > kBktK)
        for (int e = __ldcg(&ob.head[slot]); e >= 0 && !later && guard-- > 0; e = __ldcg(&ob.cand_next[e])) {
          const uint64_t eo = __ldcg(&ob.cand_order[e]);
          if (eo > my_order && (int)(eo & ((1u << kOrderStepBits) - 1)) < __ldcg(&f.L[(int)(eo >> kOrderStepBits)])) later = true;
        }
      if (!later) ob.table[slot] = (uint32_t)(v >> kSetBits);
    }
  }
}

// fast.cpp:110-141 for the steps that survived the observed-set logic: block allocation + update records (one thread per ray)
__device__ __forceinline__ void fast_emit(const FastFrame& f, int n_cast) {
  const DevCfg& cfg = f.cfg;
  const int threads_total = gridDim.x * blockDim.x;
  const int rounds = (n_cast + threads_total - 1) / threads_total;
  const int gt = ((((threadIdx.x >> 5) * gridDim.x + blockIdx.x) << 5) | (threadIdx.x & 31));   // CTA-balanced, see k_fast_solve
  for (int it = 0; it < rounds; ++it) {                     // every lane takes part in the warp-aggregated allocation
    const int r = it * threads_total + gt;
    const int U = (r < n_cast) ? __ldcg(&f.L[r]) : 0;
    const long long base = (long long)warp_alloc(&f.cnt->n_records, (unsigned long long)(U > 0 ? U : 0));
    if (U <= 0) continue;
    if (base + U > f.rec_cap) { set_err(f.cnt, 4); continue; }
    const float4 p = f.ray_param[r];
    Dda d;
    raycaster_init(d, f3(f.T.tx, f.T.ty, f.T.tz), f3(p.x, p.y, p.z), (f.ray_flags[r] & 2) != 0, cfg.carving != 0, cfg.max_ray, cfg.vsi,
                   cfg.tp.trunc, false);
    I3 last_b; last_b.x = last_b.y = last_b.z = 0x7fffffff;
    int htpos = -1;
    for (int s = 0; s < U; ++s) {
      const I3 g = dda_next(d);
      const I3 b = block_of_voxel(g, cfg.vps_inv);
      if (b.x != last_b.x || b.y != last_b.y || b.z != last_b.z) {
        last_b = b;
        if (!key_in_range(b)) { set_err(f.cnt, 5); htpos = -1; }
        else htpos = ht_find_or_insert(f.map, pack_key(b), f.cnt);
      }
      f.rec[base + s] = (htpos >= 0) ? make_record(cfg, htpos, g, (uint32_t)r) : ~0ull;
    }
  }
}

// SemanticVoxel / TsdfVoxel default construction of the frame's new blocks (semantic_voxel.h:14-27), all CTAs
__device__ __forceinline__ void fast_block_init(const FastFrame& f, int n_new, int pool_base) {
  const DevCfg& cfg = f.cfg;
  const MapRef& map = f.map;
  const int per_block = cfg.tiles_per_block;
  for (long long w = blockIdx.x; w < (long long)n_new * per_block; w += gridDim.x) {
    const int i = (int)(w / per_block), tile = (int)(w % per_block);
    const int slot = pool_base + i;
    if (slot >= map.max_blocks) { if (tile == 0 && threadIdx.x == 0) set_err(f.cnt, 3); continue; }
    if (tile == 0 && threadIdx.x == 0) {
      const int pos = map.new_list[i];
      map.ht_slot[pos] = slot;
      map.slot_key[slot] = map.ht_keys[pos];
    }
    uint8_t* chunk = map.pool + (uint64_t)slot * cfg.block_stride + (uint64_t)tile * cfg.tile_stride;
    float* dist = (float*)chunk;
    float* wgt = (float*)(chunk + cfg.plane_f32);
    uint32_t* rgba = (uint32_t*)(chunk + 2 * cfg.plane_f32);
    uint32_t* srgba = (uint32_t*)(chunk + 3 * cfg.plane_f32);
    uint8_t* label = chunk + 4 * cfg.plane_f32;
    float* prior = (float*)(chunk + cfg.head_bytes);
    const int V = cfg.tile_voxels;
    for (int v = threadIdx.x; v < V; v += blockDim.x) { dist[v] = 0.0f; wgt[v] = 0.0f; rgba[v] = 0u; srgba[v] = 0xFF7F7F7Fu; label[v] = 0; }
    for (int t = threadIdx.x; t < cfg.C * V; t += blockDim.x) prior[t] = (float)-0.60205999132;
  }
}

__global__ void __launch_bounds__(kSolveThreads, 1) k_fast_solve(FastFrame f, int max_sweeps) {
  unsigned int epoch = 0;
  unsigned int* bar = &f.fc->gridbar;
  // thread id for the item loops: consecutive 32-item chunks go to DIFFERENT CTAs (warp w of CTA b takes chunk w * gridDim.x + b),
  // so that a phase with fewer items than threads still uses every SM
  const int lane = threadIdx.x & 31;
  const int gtid = (((threadIdx.x >> 5) * gridDim.x + blockIdx.x) << 5) | lane;
  const int gthreads = gridDim.x * blockDim.x;
  Counters* cnt = f.cnt;
  const int n_points = cnt->n_points;
  const int n_cast = cnt->n_cast;
  int tl = 0;
  timeline_mark(f, tl++);
  // ---- phase 0: compaction of the cast points, in sequence order (= ray rank order)
  for (int base = (gtid & ~31); base < n_points; base += gthreads) {
    const int seq = base + lane;
    const bool c = seq < n_points && f.cast_flag[seq] != 0;
    const unsigned m = __ballot_sync(0xffffffffu, c);
    if (c) f.cast_seq[f.warp_off[seq >> 5] + __popc(m & ((1u << lane) - 1u))] = seq;
  }
  if (gtid == 0) {   // sweep ids stay monotonic across frames (slot stamps); the first sweep's counter slot was zeroed by the frame reset
    int sb = f.fc->sweep_base;
    sb = (sb + 4) & ~3;
    f.fc->sweep_base = sb;
  }
  solve_barrier(bar, epoch);
  timeline_mark(f, tl++);
  // ---- phase 1: ray set-up (first kH0 steps of every ray)
  for (int r0 = (gtid & ~31); r0 < n_cast; r0 += gthreads) fast_ray_setup(f, r0 + lane, n_cast);
  solve_barrier(bar, epoch);
  timeline_mark(f, tl++);
  // ---- phase 2: observed-set fixpoint
  const int first_sweep = ((volatile int*)&f.fc->sweep_base)[0] + 1;
  int last = first_sweep;
  bool converged = false;
  for (int it = 0; it < max_sweeps; ++it) {
    const int sweep = first_sweep + it;
    last = sweep;
    eval_sweep_body(f.cfg, cnt, f.set_offset, f.ob, f.nsteps, f.H, f.L, f.ray_state, f.ext_off, f.eval_sweep, sweep);
    solve_barrier(bar, epoch);
    if (tl < kTimelineSlots - 12) timeline_mark(f, tl++);
    const int changed = ((volatile int*)cnt->changed)[sweep & 3];
    const int err = ((volatile int*)&cnt->err)[0];
    if (!changed || err) { converged = !changed; break; }
  }
  if (gtid == 0) {
    cnt->last_sweep = last;
    f.fc->sweep_base = last;
    f.fc->sweeps_last = last - first_sweep + 1;
    if (!converged && !((volatile int*)&cnt->err)[0]) set_err(cnt, 2 /*KSG_ERR_CUDA: the solver did not converge*/);
    if (f.profile) f.fc->timeline[kTimelineSlots - 1] = tl;   // index of the first mark after the sweeps
  }
  tl = kTimelineSlots - 12;
  timeline_mark(f, tl++);
  if (((volatile int*)&cnt->err)[0] == 0 && converged) {
    // ---- phase 3: persistent table commit + ray emit (independent of each other)
    fast_obs_commit(f, n_cast);
    fast_emit(f, n_cast);
  }
  solve_barrier(bar, epoch);
  timeline_mark(f, tl++);
  const bool ok = ((volatile int*)&cnt->err)[0] == 0;
  const long long n_rec = ok ? (long long)((volatile unsigned long long*)&cnt->n_records)[0] : 0;
  // ---- phase 4: records per tile; the first record of a tile registers it
  for (long long i = gtid; i < n_rec; i += gthreads) {
    const uint64_t k = f.rec[i];
    if (k == ~0ull) continue;
    const uint32_t tk = (uint32_t)(k >> 32);
    if (atomicAdd(&f.tile_cnt[tk], 1) == 0) {
      const int idx = atomicAdd(&f.fc->n_tile_list, 1);
      if (idx < f.tile_cap) { f.tile_list[idx].tk = tk; f.tile_slot[tk] = idx; } else set_err(cnt, 4);
    }
  }
  const int n_new_raw = ((volatile int*)&cnt->n_new_blocks)[0];
  const int n_new = n_new_raw < f.map.new_cap ? n_new_raw : f.map.new_cap;
  const int pool_base = ((volatile int*)&cnt->pool_count)[0];
  solve_barrier(bar, epoch);
  timeline_mark(f, tl++);
  // ---- phase 5: key segment per tile, updated() bookkeeping, ownership (spatial sharding), new blocks
  const int n_tiles = min((long long)((volatile int*)&f.fc->n_tile_list)[0], f.tile_cap);
  for (int base = (gtid & ~31); base < n_tiles; base += gthreads) {
    const int idx = base + lane;
    int n = 0;
    uint32_t tk = 0;
    if (idx < n_tiles) { tk = f.tile_list[idx].tk; n = __ldcg(&f.tile_cnt[tk]); }
    const long long off = (long long)warp_alloc(&f.fc->rec_cursor, (unsigned long long)n);
    if (idx < n_tiles) {
      const int pos = (int)(tk / (uint32_t)f.cfg.tiles_per_block);
      const int old = atomicExch(&f.map.touched_stamp[pos], f.frame_stamp);
      if (old != f.frame_stamp) f.map.touched_list[atomicAdd(&cnt->n_blocks_touched, 1)] = pos;
      const bool owned = f.cfg.shard_count <= 1 ||
                         tile_owner(f.map.ht_keys[pos], (int)(tk % (uint32_t)f.cfg.tiles_per_block), f.cfg.shard_count) == f.cfg.shard_rank;
      f.tile_list[idx].n = owned ? n : -n;
      f.tile_list[idx].off = off;
    }
  }
  if (ok) fast_block_init(f, n_new, pool_base);
  solve_barrier(bar, epoch);
  timeline_mark(f, tl++);
  // ---- phase 6: scatter the records into their tile's segment (the counter runs back to zero: nothing to clear next frame)
  for (long long i = gtid; i < n_rec; i += gthreads) {
    const uint64_t k = f.rec[i];
    if (k == ~0ull) continue;
    const uint32_t tk = (uint32_t)(k >> 32);
    const int c = atomicSub(&f.tile_cnt[tk], 1) - 1;
    const int idx = __ldcg(&f.tile_slot[tk]);
    if (idx >= 0 && idx < n_tiles) f.keys[__ldcg(&f.tile_list[idx].off) + c] = (uint32_t)k;
  }
  if (gtid == 0) {
    int add = n_new;
    if (pool_base + add > f.map.max_blocks) add = f.map.max_blocks - pool_base;
    if (ok) cnt->pool_count = pool_base + (add > 0 ? add : 0);
    cnt->n_tiles = n_tiles;
    f.fc->tile_cursor = 0;
    f.fc->n_tile_list = 0;
    f.fc->rec_cursor = 0;
  }
  timeline_mark(f, tl++);
}

// ---------------------------------------------------------------------------------------------
// k_tile_apply_fast
// ---------------------------------------------------------------------------------------------
// ascending sort of a[0..n) by one CTA; bitonic network in its "flip" form (every compare-exchange puts the minimum at the lower
// index), so the virtual +inf padding behind n never has to move and pairs that reach past n are skipped
__device__ __forceinline__ void cta_sort_u32(uint32_t* a, int n) {
  int n2 = 1;
  while (n2 < n) n2 <<= 1;
  const int half = n2 >> 1;
  for (int k = 2; k <= n2; k <<= 1) {
    const int hk = k >> 1;
    for (int t = threadIdx.x; t < half; t += blockDim.x) {
      const int blk = t / hk, o = t - blk * hk;
      const int i = blk * k + o, p = blk * k + (k - 1 - o);
      if (p < n) { const uint32_t x = a[i], y = a[p]; if (x > y) { a[i] = y; a[p] = x; } }
    }
    __syncthreads();
    for (int j = k >> 2; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < half; t += blockDim.x) {
        const int i = (t / j) * 2 * j + (t % j), p = i + j;
        if (p < n) { const uint32_t x = a[i], y = a[p]; if (x > y) { a[i] = y; a[p] = x; } }
      }
      __syncthreads();
    }
  }
}

template <bool USE_TMA, int NCH>
__global__ void __launch_bounds__(512, 1) k_tile_apply_fast(FastFrame f, ApplySrc src) {
  extern __shared__ __align__(128) uint8_t smem[];
  const DevCfg& cfg = f.cfg;
  const int V = cfg.tile_voxels;
  const int C = cfg.C;
  float* s_dist = (float*)smem;
  float* s_wgt = (float*)(smem + cfg.plane_f32);
  uint32_t* s_rgba = (uint32_t*)(smem + 2 * cfg.plane_f32);
  uint32_t* s_srgba = (uint32_t*)(smem + 3 * cfg.plane_f32);
  uint8_t* s_label = smem + 4 * cfg.plane_f32;
  float* s_prior = (float*)(smem + cfg.head_bytes);             // only when cfg.full_stage
  const uint32_t stage_bytes = cfg.head_bytes + (cfg.full_stage ? cfg.prior_bytes : 0u);
  uint8_t* aux = smem + stage_bytes;
  int* s_seg_lo = (int*)aux;                 // [V]
  int* s_seg_hi = s_seg_lo + V;              // [V]
  uint64_t* s_bar = (uint64_t*)(s_seg_hi + V + (V & 1));
  uint32_t* s_keys = (uint32_t*)(s_bar + 2); // [kFastKeyCap]
  uint16_t* s_vox = (uint16_t*)(s_keys + kFastKeyCap);   // [V] touched voxels
  float4* s_par = (float4*)(((uintptr_t)(s_vox + V) + 15) & ~(uintptr_t)15);   // [kFastPref] operands of the sorted records
  uint32_t* s_col = (uint32_t*)(s_par + kFastPref);
  uint8_t* s_lab = (uint8_t*)(s_col + kFastPref);
  uint32_t* s_keys2 = (uint32_t*)(((uintptr_t)(s_lab + kFastPref) + 15) & ~(uintptr_t)15);   // [kFastKeyCap] records grouped by voxel
  __shared__ uint8_t s_perm[16 * 32];
  __shared__ uint8_t* s_chunk;
  __shared__ int s_g0x, s_g0y, s_g0z, s_tile, s_vox_cursor, s_nvox, s_n, s_bx, s_by, s_bz, s_log_base;
  __shared__ long long s_off;

  const int tid = threadIdx.x, lane = tid & 31;
  const int nthreads = blockDim.x;
  uint32_t phase = 0;
  if (USE_TMA && tid == 0) { mbar_init(s_bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
  __syncthreads();
  const int n_tiles = f.cnt->n_tiles;
  const F3 origin = f3(f.T.tx, f.T.ty, f.T.tz);
  const bool keep_blend = cfg.color_mode == 0;
  const uint32_t ord_mask = (1u << kRecOrdBits) - 1u;

  for (;;) {
    if (tid == 0) s_tile = atomicAdd(&f.fc->tile_cursor, 1);
    __syncthreads();
    const int j = s_tile;
    if (j >= n_tiles) break;
    if (tid == 0) {
      const TileDesc td = f.tile_list[j];
      const uint32_t tk = td.tk;
      const int pos = (int)(tk / (uint32_t)cfg.tiles_per_block), tile = (int)(tk % (uint32_t)cfg.tiles_per_block);
      const int slot = f.map.ht_slot[pos];
      uint8_t* chunk = (td.n > 0 && slot >= 0 && slot < f.map.max_blocks) ? f.map.pool + (uint64_t)slot * cfg.block_stride + (uint64_t)tile * cfg.tile_stride : nullptr;
      s_chunk = chunk;
      s_n = td.n; s_off = td.off;
      const I3 bi = unpack_key(f.map.ht_keys[pos]);
      const int tps = cfg.tiles_per_side;
      const int tx = tile % tps, ty = (tile / tps) % tps, tz = tile / (tps * tps);
      s_g0x = bi.x * cfg.vps + tx * cfg.tile_side;
      s_g0y = bi.y * cfg.vps + ty * cfg.tile_side;
      s_g0z = bi.z * cfg.vps + tz * cfg.tile_side;
      s_bx = bi.x; s_by = bi.y; s_bz = bi.z;
      s_vox_cursor = 0; s_nvox = 0;
      if (USE_TMA && chunk) { mbar_expect_tx(s_bar, stage_bytes); tma_load_1d(smem, chunk, stage_bytes, s_bar); }
    }
    __syncthreads();
    uint8_t* chunk = s_chunk;
    if (chunk == nullptr) continue;          // not owned by this shard / pool overflow already flagged
    const int n = s_n;
    // The tile's records, grouped by voxel and, inside a voxel, in ray-rank order = the reference's per-voxel update order (overlaps
    // the bulk load).  Usual case (n <= kFastKeyCap): counting sort by voxel in shared memory - histogram, scan, scatter: three barriers -
    // and the few records of one voxel are ordered by the warp that applies them.  Oversized tiles: bitonic sort in global memory.
    uint32_t* keys = f.keys + s_off;
    const bool grouped = n <= kFastKeyCap;
    bool pref = false;
    if (grouped) {
      for (int v = tid; v < V; v += nthreads) s_seg_lo[v] = 0;
      for (int i = tid; i < n; i += nthreads) s_keys[i] = keys[i];
      __syncthreads();
      for (int i = tid; i < n; i += nthreads) atomicAdd(&s_seg_lo[s_keys[i] >> kRecOrdBits], 1);
      __syncthreads();
      if (tid < 32) {        // exclusive scan of the V counts by one warp; the touched voxels are listed on the way
        const int per = (V + 31) / 32;
        const int v0 = lane * per, v1 = min(V, v0 + per);
        int local = 0;
        for (int v = v0; v < v1; ++v) local += s_seg_lo[v];
        int incl = local;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        int run = incl - local;
        for (int v = v0; v < v1; ++v) {
          const int c = s_seg_lo[v];
          s_seg_lo[v] = run; s_seg_hi[v] = run;
          if (c > 0) s_vox[atomicAdd(&s_nvox, 1)] = (uint16_t)v;
          run += c;
        }
      }
      __syncthreads();
      for (int i = tid; i < n; i += nthreads) { const uint32_t k = s_keys[i]; s_keys2[atomicAdd(&s_seg_hi[k >> kRecOrdBits], 1)] = k; }
      __syncthreads();
      keys = s_keys2;
      pref = n <= kFastPref;      // one parallel gather instead of a dependent L2 round trip per voxel
      if (pref) for (int i = tid; i < n; i += nthreads) {
        const uint32_t ord = keys[i] & ord_mask;
        s_par[i] = src.param[ord];
        s_lab[i] = src.label[ord];
        if (keep_blend) s_col[i] = src.color[ord];
      }
    } else {
      __syncthreads();
      cta_sort_u32(keys, n);
      for (int i = tid; i < n; i += nthreads) {
        const int vx = (int)(keys[i] >> kRecOrdBits);
        if (i == 0 || (int)(keys[i - 1] >> kRecOrdBits) != vx) { s_seg_lo[vx] = i; s_vox[atomicAdd(&s_nvox, 1)] = (uint16_t)vx; }
        if (i + 1 == n || (int)(keys[i + 1] >> kRecOrdBits) != vx) s_seg_hi[vx] = i + 1;
      }
    }
    if (USE_TMA) { mbar_wait(s_bar, phase); phase ^= 1; }
    else for (uint32_t t = tid; t < stage_bytes / 16; t += nthreads) ((uint4*)smem)[t] = ((const uint4*)chunk)[t];
    __syncthreads();
    float* g_prior = (float*)(chunk + cfg.head_bytes);
    const int nvox = s_nvox;
    if (f.log_head != nullptr) {   // one range of the update log per tile
      if (tid == 0) s_log_base = atomicAdd(&f.fc->log_count, nvox);
      __syncthreads();
    }
    for (;;) {
      int item = 0;
      if (lane == 0) item = atomicAdd(&s_vox_cursor, 1);
      item = __shfl_sync(0xffffffffu, item, 0);
      if (item >= nvox) break;
      const int v = s_vox[item];
      const int lo = s_seg_lo[v], hi = s_seg_hi[v];
      const int ts = cfg.tile_side_log2, tm = cfg.tile_side - 1;
      I3 g; g.x = s_g0x + (v & tm); g.y = s_g0y + ((v >> ts) & tm); g.z = s_g0z + (v >> (2 * ts));
      const F3 center = voxel_center(g, cfg.voxel_size);
      float dist = s_dist[v], wgt = s_wgt[v];
      uint32_t rgba = s_rgba[v];
      float* prow = (cfg.full_stage ? s_prior : g_prior) + (size_t)v * C;
      float p[NCH];
#pragma unroll
      for (int q = 0; q < NCH; ++q) { const int c = q * 32 + lane; p[q] = (c < C) ? prow[c] : 0.0f; }
      // order the voxel's records by ray rank (grouped tiles only; the bitonic path is sorted already)
      bool vpref = pref;
      int perm_src = lane;                        // position (relative to lo) of the record that lane handles
      if (grouped && hi - lo > 1) {
        if (hi - lo <= 32) {                      // rank sort inside the warp
          const int len = hi - lo;
          const uint32_t mine = (lane < len) ? keys[lo + lane] : 0xFFFFFFFFu;
          int rank = 0;
          for (int jj = 0; jj < len; ++jj) { const uint32_t kj = __shfl_sync(0xffffffffu, mine, jj); rank += (kj < mine) ? 1 : 0; }
          uint8_t* perm = s_perm + (tid >> 5) * 32;
          if (lane < len) perm[rank] = (uint8_t)lane;
          __syncwarp();
          if (lane < len) perm_src = perm[lane];
          __syncwarp();
        } else {                                  // long segment (rare in `fast`): in place, operands gathered from global memory
          int n2 = 1;
          const int len = hi - lo;
          uint32_t* a = keys + lo;
          while (n2 < len) n2 <<= 1;
          const int half = n2 >> 1;
          for (int k = 2; k <= n2; k <<= 1) {
            const int hk = k >> 1;
            for (int t = lane; t < half; t += 32) {
              const int blk = t / hk, o = t - blk * hk;
              const int i = blk * k + o, pp = blk * k + (k - 1 - o);
              if (pp < len) { const uint32_t x = a[i], y = a[pp]; if (x > y) { a[i] = y; a[pp] = x; } }
            }
            __syncwarp();
            for (int jx = k >> 2; jx > 0; jx >>= 1) {
              for (int t = lane; t < half; t += 32) {
                const int i = (t / jx) * 2 * jx + (t % jx), pp = i + jx;
                if (pp < len) { const uint32_t x = a[i], y = a[pp]; if (x > y) { a[i] = y; a[pp] = x; } }
              }
              __syncwarp();
            }
          }
          vpref = false;
        }
      }
      for (int base = lo; base < hi; base += 32) {
        const int k = (hi - lo <= 32) ? lo + perm_src : base + lane;
        uint32_t ord = 0, col = 0;
        int lab = 0;
        float sdf = 0.0f, uw = 0.0f;
        if (base + lane < hi) {
          ord = keys[k] & ord_mask;
          const float4 pr = vpref ? s_par[k] : src.param[ord];
          tsdf_measure(cfg.tp, origin, f3(pr.x, pr.y, pr.z), center, pr.w, sdf, uw);
          if (keep_blend) col = vpref ? s_col[k] : src.color[ord];
          lab = vpref ? (int)s_lab[k] : (int)src.label[ord];
        }
        const int nb = (hi - base) < 32 ? (hi - base) : 32;
        for (int jj = 0; jj < nb; ++jj) {      // semantic rows: lanes = classes, one-hot frequencies (fast.cpp:132-135)
          const int l = __shfl_sync(0xffffffffu, lab, jj);
          if (l != 0) {   // label 0: column 0 of the likelihood is zero (base.cpp:127)
#pragma unroll
            for (int q = 0; q < NCH; ++q) p[q] += ((q * 32 + lane) == l) ? cfg.lm : cfg.ln;
          }
        }
        tsdf_batch(cfg.tp, lane, nb, sdf, uw, col, keep_blend, dist, wgt, rgba);
      }
      // arg-max, first maximum wins (base.cpp:352-367)
      float best = -3.402823466e38f;
      int bi = 0x7fffffff;
#pragma unroll
      for (int q = 0; q < NCH; ++q) { const int c = q * 32 + lane; if (c < C && (p[q] > best || bi == 0x7fffffff)) { best = p[q]; bi = c; } }
      for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_down_sync(0xffffffffu, best, o);
        const int oi = __shfl_down_sync(0xffffffffu, bi, o);
        if (oi != 0x7fffffff && (bi == 0x7fffffff || ob > best || (ob == best && oi < bi))) { best = ob; bi = oi; }
      }
      best = __shfl_sync(0xffffffffu, best, 0);
      const int bi_lab = __shfl_sync(0xffffffffu, bi, 0);
#pragma unroll
      for (int q = 0; q < NCH; ++q) { const int c = q * 32 + lane; if (c < C) prow[c] = p[q]; }
      if (lane == 0) {
        s_dist[v] = dist; s_wgt[v] = wgt;
        s_label[v] = (uint8_t)bi_lab;
        const uint32_t sc = f.luts->label_rgba[bi_lab];          // base.cpp:370-380
        s_srgba[v] = sc;
        if (cfg.color_mode == 1) s_rgba[v] = sc;                 // kSemantic (base.cpp:177-180)
        else if (cfg.color_mode == 2) s_rgba[v] = rainbow_color_map((double)expf(best));  // base.cpp:181-185
        else s_rgba[v] = rgba;                                   // kColor: the blended colour is the result
      }
      if (f.log_head != nullptr) {
        const int at = s_log_base + item;
        if (at < f.log_cap) {
          if (lane == 0) {
            const int m = cfg.vps - 1;
            VoxelUpdate u;
            u.bx = s_bx; u.by = s_by; u.bz = s_bz;
            u.lin_label = (uint32_t)((g.x & m) + cfg.vps * ((g.y & m) + cfg.vps * (g.z & m))) | ((uint32_t)bi_lab << 24);
            u.dist = dist; u.wgt = wgt; u.rgba = s_rgba[v]; u.srgba = s_srgba[v];
            f.log_head[at] = u;
          }
#pragma unroll
          for (int q = 0; q < NCH; ++q) { const int c = q * 32 + lane; if (c < C) f.log_prior[(size_t)at * C + c] = p[q]; }
        }
      }
    }
    if (USE_TMA) {
      fence_proxy_async();
      __syncthreads();
      if (tid == 0) { tma_store_1d(chunk, smem, stage_bytes); tma_store_commit_wait(); }
    } else {
      __syncthreads();
      for (uint32_t t = tid; t < stage_bytes / 16; t += nthreads) ((uint4*)chunk)[t] = ((const uint4*)smem)[t];
    }
    // the loop-top barrier orders the store's completion before the next tile's load
  }
}

}  // namespace ksg
