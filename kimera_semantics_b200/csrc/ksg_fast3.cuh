// ksg_fast3.cuh — observed-set solver, third formulation (round 2), used by k_fast_solve3.
//
// What the first measurements of the persistent kernel showed (profiles/r02/bench_fast5_v2.json: sweeps of 90 / 81 / 54 / 20 us):
//   * sweep 1 starts from "nothing but the guaranteed first steps is performed", so nearly every ray runs its full length
//     (~1.9 M candidate steps materialised for ~57 K final updates), and sweep 2 takes almost all of it back;
//   * every ray that toggles a slot re-evaluates itself in the next sweep (it sees its own stamp);
//   * per candidate the solver chased four arrays (value, order, position, link).
// Changes, none of which alters the fixpoint (DESIGN.md section 4: the dependency is triangular in rank order, the fixpoint unique):
//   1. RANK GROUPS.  A ray depends only on rays of lower rank, so once ranks [0, n) have converged they are FINAL whatever the
//      higher ranks do.  Rays are solved in groups of growing size (512, then x4); a group iterates to convergence against the
//      finished lower groups.  With the `mixed` order the low ranks are a uniform sub-sample of the image, so a new group already
//      sees most of the free space carved: its first evaluation is close to the answer, finished groups are never polled again.
//   2. one 16-byte record per candidate {packed voxel index, bucket position, sweep of the owner's last toggle} and one per ray
//      {materialised steps, updates, length, last evaluation}: one load each; the set value (hash + offset) is recomputed from the
//      voxel index; flipping a candidate's "performed" bit is a plain store (the owner knows the whole entry).
//   3. the per-slot stamp is (sweep << 8 | toggles in that sweep): a ray is NOT dirty when the only toggle of the slot in its last
//      sweep was its own.
//   4. no record buffer: after convergence the performed candidates are walked twice, fully parallel (8 lanes per ray):
//      pass 1 commits the persistent table, allocates blocks and counts records per tile; pass 2 writes the (voxel, rank) keys
//      straight into the tile's segment.  The voxel index kept per candidate replaces the second ray walk.
#pragma once
#include "ksg_fast.cuh"

namespace ksg {

struct __align__(16) Cand { uint64_t vkey; int pos; int tog; };      // pos: >= 0 bucket entry, -2 not inserted, <= -3 overflow entry -3-pos
struct __align__(16) OvfEnt { uint64_t order_perf; uint32_t hi; int next; };
struct __align__(16) RayRec { int H, L, nsteps, eval_sweep; };
static constexpr int kBkt3 = 32;              // bucket entries per approximate-set slot (256 B): systematic aliases of the index hash stack 2-3 voxels per slot
static constexpr int kOvfPending = -2;        // overflow entry published, link not yet written
static constexpr int kSortPerWarp = 1024;     // visitors of a shared start-set slot sorted in shared memory (more: in place in global memory)

__device__ __forceinline__ Cand ld_cand(const Cand* p) {
  const int4 v = __ldcg((const int4*)p);
  Cand c; c.vkey = ((uint64_t)(uint32_t)v.y << 32) | (uint32_t)v.x; c.pos = v.z; c.tog = v.w;
  return c;
}
__device__ __forceinline__ void st_cand(Cand* p, uint64_t vkey, int pos, int tog) {
  __stcg((int4*)p, make_int4((int)(uint32_t)vkey, (int)(uint32_t)(vkey >> 32), pos, tog));
}
__device__ __forceinline__ void st_cand_state(Cand* p, int pos, int tog) { __stcg((int2*)p + 1, make_int2(pos, tog)); }
__device__ __forceinline__ uint64_t cand_value(uint64_t vkey, uint64_t offset) { return (uint64_t)index_hash(unpack_key(vkey)) + offset; }
__device__ __forceinline__ uint64_t make_entry(bool on, uint64_t order, uint64_t v) { return (on ? kEntPerf : 0ull) | (order << 13) | (v >> kSetBits); }
__device__ __forceinline__ long long cand_index3(const Obs3& o, const long long* ext_off, int r, int s) {
  if (s < kH0) return (long long)r * kH0 + s;
  const int k = 31 - __clz(s >> 4);
  return o.ext_base + __ldcg(&ext_off[(size_t)r * kExtSegs + k]) + (s - (kH0 << k));
}

// A toggle of `slot` by ray r in sweep k leaves (k, r) in two monotonic words: smax = max (k << 32 | r), smin = min ((~k) << 32 | r).
// Both are fire-and-forget reductions.  A ray evaluated last in sweep `last` is dirty iff the slot was toggled in a later sweep, or in
// sweep `last` by a ray other than itself (smallest and largest toggler of that sweep are not both the ray).
static constexpr uint32_t kSweepCap = 0x7FFFFFFFu;
__device__ __forceinline__ void stamp_toggle(const Obs3& o, uint32_t slot, int sweep, int r) {
  atomicMax((unsigned long long*)&o.stamp_max[slot], ((unsigned long long)(uint32_t)sweep << 32) | (uint32_t)r);
  atomicMin((unsigned long long*)&o.stamp_min[slot], ((unsigned long long)(kSweepCap - (uint32_t)sweep) << 32) | (uint32_t)r);
}
__device__ __forceinline__ bool stamp_dirty(const Obs3& o, uint32_t slot, int last, int r) {
  const unsigned long long a = __ldcg((const unsigned long long*)&o.stamp_max[slot]);
  const unsigned long long b = __ldcg((const unsigned long long*)&o.stamp_min[slot]);
  const int sk = (int)(a >> 32);
  if (sk > last) return true;
  if (sk < last) return false;
  return !((uint32_t)(b >> 32) == kSweepCap - (uint32_t)sk && (uint32_t)a == (uint32_t)r && (uint32_t)b == (uint32_t)r);
}

// first time a candidate turns performed: it enters the slot's bucket (or the overflow pool); returns its position code.
// The overflow push is one exchange, no retry loop and no fence: a reader that catches the entry half-written (pending link, fields of
// an older frame) takes a wrong decision for this sweep only - the inserter stamps the slot afterwards, which marks that reader dirty.
__device__ __forceinline__ int cand_insert3(const FastFrame& f, uint32_t slot, uint64_t entry) {
  const Obs3& o = f.o3;
  const int idx = atomicAdd(&o.slot_cnt[slot], 1);
  if (f.profile) dbg_max(f, 16, idx + 1);
  if (idx < kBkt3) { const int pos = (int)slot * kBkt3 + idx; __stcg(&o.bkt[pos], entry); return pos; }
  const int id = atomicAdd(&f.fc->ovf_count, 1);
  if (id >= o.ovf_cap) { set_err(f.cnt, 4); return -2; }
  OvfEnt* e = &o.ovf[id];
  __stcg(&e->next, kOvfPending);
  __stcg(&e->order_perf, (entry & kEntPerf) | ((entry >> 13) & ((1ull << kEntOrderBits) - 1)));
  __stcg(&e->hi, (uint32_t)(entry & 0x1FFFull));
  const int old = atomicExch(&o.head[slot], id);
  __stcg(&e->next, old);
  return -3 - id;
}

// latest performed visit of `slot` that precedes `my_order`: its (value >> 20), or -1.  (A non-inlined variant of these helpers was measured
// 20 % slower on the whole frame - profiles/r02/bench_full_9.json - so they stay inline; the loops past the first 8 entries are rolled.)
__device__ __forceinline__ int latest_performed_before_raw(const uint64_t* bkt, const int* slot_cnt, const int* head, const OvfEnt* ovf, int ovf_cap,
                                                        uint32_t slot, uint64_t my_order) {
  const ulonglong2* b = (const ulonglong2*)(bkt + (size_t)slot * kBkt3);
  const int total = __ldcg(&slot_cnt[slot]);
  ulonglong2 v[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) v[q] = __ldcg(b + q);      // independent of the count: one round trip for the usual <= 8 entries
  const int n = total < kBkt3 ? total : kBkt3;
  long long best = -1;
  int best_hi = -1;
#pragma unroll
  for (int q = 0; q < 4; ++q) scan_entries(v[q], 2 * q, n, my_order, best, best_hi);
#pragma unroll 1
  for (int q0 = 4; 2 * q0 < n; q0 += 4) {
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = __ldcg(b + q0 + q);
#pragma unroll
    for (int q = 0; q < 4; ++q) scan_entries(v[q], 2 * (q0 + q), n, my_order, best, best_hi);
  }
  if (total > kBkt3) {
    int guard = total - kBkt3 + 8;
#pragma unroll 1
    for (int id = __ldcg(&head[slot]); id >= 0 && id < ovf_cap && guard-- > 0; id = __ldcg(&ovf[id].next)) {
      const uint64_t op = __ldcg(&ovf[id].order_perf);
      const uint64_t eo = op & ~kEntPerf;
      if ((op & kEntPerf) && eo < my_order && (long long)eo > best) { best = (long long)eo; best_hi = (int)__ldcg(&ovf[id].hi); }
    }
  }
  return best_hi;
}
__device__ __forceinline__ int latest_performed_before3(const Obs3& o, uint32_t slot, uint64_t my_order) {
  return latest_performed_before_raw(o.bkt, o.slot_cnt, o.head, o.ovf, o.ovf_cap, slot, my_order);
}
__device__ __forceinline__ bool later_performed_exists_raw(const uint64_t* bkt, const int* slot_cnt, const int* head, const OvfEnt* ovf, int ovf_cap,
                                                        uint32_t slot, uint64_t my_order) {
  // the bucket is read 8 entries (4 x 16 B) per round trip, the first 8 independently of the count, as in latest_performed_before_raw:
  // one dependent load per entry made the table commit as long as its slowest hot slot (up to 32 trips)
  const ulonglong2* b = (const ulonglong2*)(bkt + (size_t)slot * kBkt3);
  const int total = __ldcg(&slot_cnt[slot]);
  ulonglong2 v[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) v[q] = __ldcg(b + q);
  const int n = total < kBkt3 ? total : kBkt3;
  bool later = false;
#pragma unroll 1
  for (int q0 = 0;;) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint64_t e2[2] = {v[q].x, v[q].y};
#pragma unroll
      for (int k = 0; k < 2; ++k)
        if (2 * (q0 + q) + k < n && (e2[k] & kEntPerf) && ((e2[k] >> 13) & ((1ull << kEntOrderBits) - 1)) > my_order) later = true;
    }
    q0 += 4;
    if (2 * q0 >= n) break;
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = __ldcg(b + q0 + q);
  }
  if (total > kBkt3) {
    int guard = total - kBkt3 + 8;
#pragma unroll 1
    for (int id = __ldcg(&head[slot]); id >= 0 && id < ovf_cap && !later && guard-- > 0; id = __ldcg(&ovf[id].next)) {
      const uint64_t op = __ldcg(&ovf[id].order_perf);
      if ((op & kEntPerf) && (op & ~kEntPerf) > my_order) later = true;
    }
  }
  return later;
}
__device__ __forceinline__ bool later_performed_exists3(const Obs3& o, uint32_t slot, uint64_t my_order) {
  return later_performed_exists_raw(o.bkt, o.slot_cnt, o.head, o.ovf, o.ovf_cap, slot, my_order);
}

// single writer per candidate: the warp that owns the ray.  c.pos is updated when the candidate enters a bucket.
// No fence between the entry and the stamp: a reader of the same sweep that misses the entry is flagged by the stamp (another
// ray toggled its slot in its own sweep), and every store is visible after the grid barrier that ends the sweep.
__device__ __forceinline__ void set_performed3(const FastFrame& f, Cand& c, long long ci, uint32_t slot, uint64_t order, uint64_t v, bool on, int sweep, int r) {
  const Obs3& o = f.o3;
  if (c.pos >= 0) __stcg(&o.bkt[c.pos], make_entry(on, order, v));
  else if (c.pos <= -3) __stcg(&o.ovf[-3 - c.pos].order_perf, (on ? kEntPerf : 0ull) | order);
  else if (on) { c.pos = cand_insert3(f, slot, make_entry(true, order, v)); st_cand_state(&o.cand[ci], c.pos, 0); }
  else return;                       // never entered a bucket and stays unperformed: invisible to every other ray
  stamp_toggle(o, slot, sweep, r);
}

// ---------------------------------------------------------------------------------------------
// RayCaster steps (A.7) of ONE ray by a whole warp.  The serial walk picks, at every step, the axis with the smallest
// t_to_next_boundary_ (first minimum wins) and adds that axis' t_step_size_ to it: per axis the boundary times form the chain
// a(j+1) = fl(a(j) + ts), independent of the other axes, and the walk is the merge of the three non-decreasing chains ordered by
// (time, axis, index).  So: three lanes run the three chains (W dependent additions each instead of 3 W dependent steps), every
// element finds its rank with two binary searches, and the element of rank s carries the per-axis step counts before step s,
// i.e. the voxel emitted at step s.  Bit-identical to dda_next as long as every time and step is finite and every step positive
// (else the caller walks serially: NaN / zero components follow the comparison semantics of the serial code).
// ---------------------------------------------------------------------------------------------
static constexpr int kWin = 64;               // steps per window (= the evaluation block)
struct WarpDdaScratch { float a[3][kWin + 1]; int endc[4]; uint64_t out[kWin]; };

__device__ __forceinline__ bool ray_state_parallel_ok(const RayState& st) {
  const bool fin = isfinite(st.tn0) && isfinite(st.tn1) && isfinite(st.tn2) && isfinite(st.ts0) && isfinite(st.ts1) && isfinite(st.ts2);
  return fin && st.ts0 > 0.0f && st.ts1 > 0.0f && st.ts2 > 0.0f;
}
// W <= kWin steps from `st`; sc->out[0..W) = packed voxel indices, st advanced by W steps.  Returns false if an index left the packed range.
__device__ __forceinline__ bool warp_dda_window(RayState& st, int W, WarpDdaScratch* sc, int lane) {
  if (lane < 3) {
    float a = lane == 0 ? st.tn0 : (lane == 1 ? st.tn1 : st.tn2);
    const float ts = lane == 0 ? st.ts0 : (lane == 1 ? st.ts1 : st.ts2);
    sc->a[lane][0] = a;
    for (int j = 1; j <= W; ++j) { a = a + ts; sc->a[lane][j] = a; }
  }
  __syncwarp();
  const int sg0 = (st.sg & 3) - 1, sg1 = ((st.sg >> 2) & 3) - 1, sg2 = ((st.sg >> 4) & 3) - 1;
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    for (int j = lane; j <= W; j += 32) {
      const float v = sc->a[k][j];
      int cnt[3];
      cnt[k] = j;
#pragma unroll
      for (int d = 1; d < 3; ++d) {
        const int k2 = (k + d) % 3;
        const float* b = sc->a[k2];
        // elements of axis k2 that precede (v, k): value < v, or value == v when k2 < k
        int lo = 0, hi = W + 1;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          const float x = b[mid];
          const bool before = (k2 < k) ? (x <= v) : (x < v);
          if (before) lo = mid + 1; else hi = mid;
        }
        cnt[k2] = lo;
      }
      const int rank = cnt[0] + cnt[1] + cnt[2];
      if (rank <= W) {
        I3 g; g.x = st.cx + sg0 * cnt[0]; g.y = st.cy + sg1 * cnt[1]; g.z = st.cz + sg2 * cnt[2];
        if (rank < W) { if (key_in_range(g)) sc->out[rank] = pack_key(g); else ok = false; }
        else { sc->endc[0] = cnt[0]; sc->endc[1] = cnt[1]; sc->endc[2] = cnt[2]; }
      }
    }
  }
  __syncwarp();
  const int e0 = sc->endc[0], e1 = sc->endc[1], e2 = sc->endc[2];
  st.cx += sg0 * e0; st.cy += sg1 * e1; st.cz += sg2 * e2;
  st.tn0 = sc->a[0][e0]; st.tn1 = sc->a[1][e1]; st.tn2 = sc->a[2][e2];
  return __all_sync(0xffffffffu, ok);
}

// evaluation blocks: [0,16), [16,32), [32,64), then 64 steps at a time; a block never straddles a storage segment
__device__ __forceinline__ void block_of_step(int s, int& s0, int& blen) {
  if (s < kH0) { s0 = 0; blen = kH0; return; }
  const int k = 31 - __clz(s >> 4);
  const int seg = kH0 << k;
  if (seg <= kWin) { s0 = seg; blen = seg; }
  else { s0 = seg + ((s - seg) & ~(kWin - 1)); blen = kWin; }
}

__device__ __forceinline__ void fast3_ray_setup(const FastFrame& f, int r, int n_cast) {
  const DevCfg& cfg = f.cfg;
  const Obs3& o = f.o3;
  int h = 0;
  const long long t_begin = f.profile ? clock64() : 0;
  long long t_ins = 0;
  if (r < n_cast) {
    const int seq = f.cast_seq[r];
    const float4 p = f.pt_pG[seq];
    const uint8_t fl = f.pt_flags[seq];
    f.ray_param[r] = p;
    f.ray_label[r] = f.pt_label[seq];
    f.ray_flags[r] = fl;
    f.ray_color[r] = f.pt_color[seq];
    if (f.profile) dbg_max(f, 12, clock64() - t_begin);
    Dda d;
    raycaster_init(d, f3(f.T.tx, f.T.ty, f.T.tz), f3(p.x, p.y, p.z), (fl & 2) != 0, cfg.carving != 0, cfg.max_ray, cfg.vsi, cfg.tp.trunc,
                   /*cast_from_origin=*/false);
    int n = d.length_in_steps + 1;
    if (!d.in_range || n >= (1 << kOrderStepBits)) { set_err(f.cnt, 5); n = 0; }
    if (f.profile) dbg_max(f, 13, clock64() - t_begin);
    h = n < kH0 ? n : kH0;
    const int l0 = h < cfg.maxc ? h : cfg.maxc;   // a ray cannot break before `maxc` consecutive collisions
    for (int s = 0; s < h; ++s) {
      const I3 g = dda_next(d);
      if (!key_in_range(g)) { set_err(f.cnt, 5); h = s; break; }
      const uint64_t vkey = pack_key(g);
      const long long ci = (long long)r * kH0 + s;
      int pos = -2;
      if (s < l0) {
        const long long t0 = f.profile ? clock64() : 0;
        const uint64_t v = (uint64_t)index_hash(g) + f.set_offset;
        pos = cand_insert3(f, (uint32_t)v & kSetMask, make_entry(true, ((uint64_t)r << kOrderStepBits) | (uint64_t)s, v));
        if (f.profile) t_ins += clock64() - t0;
      }
      st_cand(&o.cand[ci], vkey, pos, 0);
    }
    if (f.profile) dbg_max(f, 14, clock64() - t_begin);
    RayState st; save_state(st, d); f.ray_state[r] = st;
    RayRec rr; rr.H = h; rr.L = (h < l0) ? h : l0; rr.nsteps = (h < kH0 && h < n) ? h : n; rr.eval_sweep = 0;
    *(int4*)&f.rayrec[r] = make_int4(rr.H, rr.L, rr.nsteps, rr.eval_sweep);
  }
  warp_add(&f.cnt->ray_steps, (unsigned long long)h);
  if (f.profile) { dbg_max(f, 0, clock64() - t_begin); dbg_max(f, 1, t_ins); }
}

// One sweep over the rays [r_lo, r_hi): one warp per ray.  A ray is re-evaluated only from the first block that holds a dirty
// step (the consecutive-collision count at every block start is kept), in blocks of up to 64 steps = two steps per lane; steps that
// do not exist yet are produced by the warp-parallel ray walk.
__device__ __forceinline__ void fast3_sweep(const FastFrame& f, int sweep, int r_lo, int r_hi, WarpDdaScratch* sc) {
  const Obs3& o = f.o3;
  const DevCfg& cfg = f.cfg;
  Counters* cnt = f.cnt;
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  if (blockIdx.x == 0 && threadIdx.x == 0) cnt->changed[(sweep + 1) & 3] = 0;
  for (int r = r_lo + (threadIdx.x >> 5) * gridDim.x + blockIdx.x; r < r_hi; r += warps_total) {
    const int4 rr = __ldcg((const int4*)&f.rayrec[r]);
    int h = rr.x;
    const int old = rr.y, n = rr.z, last = rr.w;
    int fd = 0x7fffffff;                                        // first dirty step
    if (last == 0) fd = 0;
    else {
      const int upto = (old < h - 1) ? old : h - 1;             // steps 0..upto were examined last time
      for (int s = lane; s <= upto; s += 32) {
        const Cand c = ld_cand(&o.cand[cand_index3(o, f.ext_off, r, s)]);
        const uint32_t slot = (uint32_t)cand_value(c.vkey, f.set_offset) & kSetMask;
        if (stamp_dirty(o, slot, last, r)) { fd = s; break; }
      }
      for (int d = 16; d > 0; d >>= 1) { const int t = __shfl_xor_sync(0xffffffffu, fd, d); fd = t < fd ? t : fd; }
    }
    if (fd == 0x7fffffff) { if (f.profile && lane == 0) dbg_add(f, 18, 1); continue; }
    const long long t_eval = f.profile ? clock64() : 0;
    int n_blocks_eval = 0, n_blocks_mat = 0;
    int s0, blen;
    block_of_step(fd, s0, blen);
    long long base_ci = cand_index3(o, f.ext_off, r, s0);
    int run = (s0 == 0) ? 0 : __ldcg(&f.blk_run[base_ci >> 4]);
    int U = -1;
    while (s0 < n && U < 0) {
      const int cend = (s0 + blen < n) ? s0 + blen : n;
      ++n_blocks_eval;
      if (s0 >= h) {   // materialise the block: continue the ray walk (A.7) from the saved state
        ++n_blocks_mat;
        int ok = 1;
        if (lane == 0 && s0 >= kH0 && (s0 & (s0 - 1)) == 0) {   // s0 = 16 << k: first block of storage segment k (steps [16<<k, 32<<k))
          const int k = 31 - __clz(s0 >> 4);
          const long long need_c = s0;
          const long long off = (long long)atomicAdd(&cnt->n_cand_ext, (unsigned long long)need_c);
          if (o.ext_base + off + need_c > o.cand_cap) { set_err(cnt, 4); ok = 0; }
          else f.ext_off[(size_t)r * kExtSegs + k] = off;
        }
        ok = __shfl_sync(0xffffffffu, ok, 0);
        if (ok) {
          __syncwarp();
          base_ci = cand_index3(o, f.ext_off, r, s0);
          RayState st = f.ray_state[r];
          const int W = cend - s0;
          if (ray_state_parallel_ok(st)) {
            if (!warp_dda_window(st, W, sc, lane)) { set_err(cnt, 5); ok = 0; }
            else {
              for (int t = lane; t < W; t += 32) st_cand(&o.cand[base_ci + t], sc->out[t], -2, 0);
              if (lane == 0) f.ray_state[r] = st;
            }
            __syncwarp();
          } else {
            if (lane == 0) {
              Dda d; load_state(d, st);
              for (int t = 0; t < W; ++t) {
                const I3 g = dda_next(d);
                if (!key_in_range(g)) { set_err(cnt, 5); ok = 0; break; }
                st_cand(&o.cand[base_ci + t], pack_key(g), -2, 0);
              }
              if (ok) { save_state(st, d); f.ray_state[r] = st; }
            }
            ok = __shfl_sync(0xffffffffu, ok, 0);
            __syncwarp();
          }
          if (ok && lane == 0) { f.rayrec[r].H = cend; atomicAdd(&cnt->ray_steps, (unsigned long long)W); }
        }
        if (!ok) { U = s0; break; }   // scratch exhausted / index range (flagged): stop here
        h = cend;
      }
      if (lane == 0 && s0 > 0) f.blk_run[base_ci >> 4] = run;
      // ---- collisions of the block's steps: two per lane
      Cand c[2];
      uint64_t v[2];
      bool coll[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int s = s0 + q * 32 + lane;
        c[q].vkey = 0; c[q].pos = -2; c[q].tog = 0; v[q] = 0; coll[q] = false;
        if (s < cend) { c[q] = ld_cand(&o.cand[base_ci + q * 32 + lane]); v[q] = cand_value(c[q].vkey, f.set_offset); }
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int s = s0 + q * 32 + lane;
        if (s < cend) {
          const uint32_t slot = (uint32_t)v[q] & kSetMask;
          const uint32_t stale = o.table[slot];   // issued together with the bucket loads
          const int hi = latest_performed_before3(o, slot, ((uint64_t)r << kOrderStepBits) | (uint64_t)s);
          coll[q] = (hi >= 0) ? ((uint32_t)hi == (uint32_t)(v[q] >> kSetBits)) : (stale == (uint32_t)(v[q] >> kSetBits));
          if (f.profile) { const int tot = __ldcg(&o.slot_cnt[slot]); if (tot > kBkt3) dbg_max(f, 17, tot - kBkt3); }
        }
      }
      const unsigned bits0 = __ballot_sync(0xffffffffu, coll[0]), bits1 = __ballot_sync(0xffffffffu, coll[1]);
      if (f.profile && lane == 0 && n_blocks_eval == 1) dbg_max(f, 15, clock64() - t_eval);
      int brk = -1;
      for (int jj = 0; s0 + jj < cend; ++jj) {
        const unsigned bit = (jj < 32) ? ((bits0 >> jj) & 1u) : ((bits1 >> (jj - 32)) & 1u);
        if (bit) ++run; else run = 0;                          // fast.cpp:115-119
        if (run > cfg.maxc) { brk = s0 + jj; break; }          // fast.cpp:120-122
      }
      const int perf_end = (brk >= 0) ? brk : cend;
#pragma unroll
      for (int q = 0; q < 2; ++q) {                            // newly performed steps of this block
        const int s = s0 + q * 32 + lane;
        if (s < perf_end && s >= old)
          set_performed3(f, c[q], base_ci + q * 32 + lane, (uint32_t)v[q] & kSetMask, ((uint64_t)r << kOrderStepBits) | (uint64_t)s, v[q], true, sweep, r);
      }
      __syncwarp();
      if (brk >= 0) { U = brk; break; }
      s0 = cend;
      if (s0 < n) { int nb; block_of_step(s0, s0, nb); blen = nb; if (s0 < h) base_ci = cand_index3(o, f.ext_off, r, s0); }
    }
    if (U < 0) U = n;   // the ray ran its full length
    if (U < old) {      // steps [U, old) are no longer performed
      for (int s = U + lane; s < old; s += 32) {
        const long long ci = cand_index3(o, f.ext_off, r, s);
        Cand c = ld_cand(&o.cand[ci]);
        const uint64_t v = cand_value(c.vkey, f.set_offset);
        set_performed3(f, c, ci, (uint32_t)v & kSetMask, ((uint64_t)r << kOrderStepBits) | (uint64_t)s, v, false, sweep, r);
      }
    }
    if (lane == 0) {
      if (U != old) { f.rayrec[r].L = U; cnt->changed[sweep & 3] = 1; }
      f.rayrec[r].eval_sweep = sweep;
      if (f.profile) { dbg_max(f, 3, clock64() - t_eval); dbg_add(f, 4, 1); dbg_add(f, 5, n_blocks_eval); dbg_add(f, 6, n_blocks_mat); if (U != old) dbg_add(f, 7, 1); dbg_add(f, 19, 1); }
    }
  }
}

// The performed candidates of every ray, 8 lanes per ray.  PASS 1: persistent table commit (the last performed visit of a slot
// survives the frame), block allocation (base.cpp:205-254), records per tile.  PASS 2: (voxel, rank) key into the tile's segment.
template <int PASS>
__device__ __forceinline__ void fast3_walk_performed(const FastFrame& f, int n_cast, int n_tiles) {
  constexpr int G = 8;
  const Obs3& o = f.o3;
  const DevCfg& cfg = f.cfg;
  const int groups_total = (gridDim.x * blockDim.x) / G;
  const int gl = threadIdx.x % G;
  const int gt = ((((threadIdx.x >> 5) * gridDim.x + blockIdx.x) << 5) | (threadIdx.x & 31));   // CTA-balanced
  for (int r = gt / G; r < n_cast; r += groups_total) {
    const int U = __ldcg(&f.rayrec[r].L);
    for (int s = gl; s < U; s += G) {
      const Cand c = ld_cand(&o.cand[cand_index3(o, f.ext_off, r, s)]);
      const I3 g = unpack_key(c.vkey);
      if (PASS == 1) {
        const uint64_t v = (uint64_t)index_hash(g) + f.set_offset;
        const uint32_t slot = (uint32_t)v & kSetMask;
        if (!later_performed_exists3(o, slot, ((uint64_t)r << kOrderStepBits) | (uint64_t)s)) o.table[slot] = (uint32_t)(v >> kSetBits);
      }
      const I3 b = block_of_voxel(g, cfg.vps_inv);
      if (!key_in_range(b)) { set_err(f.cnt, 5); continue; }
      const int htpos = ht_find_or_insert(f.map, pack_key(b), f.cnt);
      if (htpos < 0) continue;
      const uint64_t rec = make_record(cfg, htpos, g, (uint32_t)r);
      const uint32_t tk = (uint32_t)(rec >> 32);
      if (PASS == 1) {
        if (atomicAdd(&f.tile_cnt[tk], 1) == 0) {
          const int idx = atomicAdd(&f.fc->n_tile_list, 1);
          if (idx < f.tile_cap) { f.tile_list[idx].tk = tk; f.tile_slot[tk] = idx; } else set_err(f.cnt, 4);
        }
      } else {
        const int at = atomicSub(&f.tile_cnt[tk], 1) - 1;
        const int idx = __ldcg(&f.tile_slot[tk]);
        if (idx >= 0 && idx < n_tiles && at >= 0) f.keys[__ldcg(&f.tile_list[idx].off) + at] = (uint32_t)rec;
      }
    }
  }
}

__global__ void __launch_bounds__(kSolveThreads, 1) k_fast_solve3(FastFrame f, int max_sweeps) {
  unsigned int epoch = 0;
  unsigned int* bar = &f.fc->gridbar;
  const int lane = threadIdx.x & 31;
  const int gtid = (((threadIdx.x >> 5) * gridDim.x + blockIdx.x) << 5) | lane;   // consecutive 32-item chunks go to different CTAs
  const int gthreads = gridDim.x * blockDim.x;
  Counters* cnt = f.cnt;
  const int n_points = cnt->n_points;
  int tl = 0;
  prof_init(f);
  timeline_mark(f, tl++);
  extern __shared__ int s_sort[];            // kSortPerWarp ints per warp
  // ---- phase 0a: start-set slots shared by several cells: every visitor files itself in the slot's list
  const int n_mixed = ((volatile int*)&f.fc->n_mixed)[0];
  if (n_mixed > 0) {
    for (int seq = gtid; seq < n_points; seq += gthreads) {
      const uint64_t v = f.pt_key[seq];
      if (v == ~0ull) continue;
      const uint32_t slot = (uint32_t)v & kSetMask;
      if (f.s_hmin[slot] != f.s_hmax[slot]) f.m_list[f.s_base[slot] + f.sb.next[seq]] = seq;
    }
    prof_flush(f, -1);
    solve_barrier(bar, epoch);
    timeline_mark(f, 57);
    // ---- phase 0b: one warp per such slot: visitors in sequence order; a visitor is cast iff its predecessor carried another value
    const int warps_total = gthreads >> 5;
    int* scratch = s_sort + (threadIdx.x >> 5) * kSortPerWarp;
    for (int mi = (threadIdx.x >> 5) * gridDim.x + blockIdx.x; mi < n_mixed; mi += warps_total) {
      const int slot = f.mixed_list[mi];
      const int n = __ldcg(&f.s_visits[slot]);
      int* seg = f.m_list + __ldcg(&f.s_base[slot]);
      int* a = seg;
      if (n <= kSortPerWarp) {
#pragma unroll 4
        for (int i = lane; i < n; i += 32) scratch[i] = __ldcg(&seg[i]);
        a = scratch;
      }
      __syncwarp();
      warp_sort_i32(a, n, lane);
      for (int i0 = 1 + lane; i0 < n; i0 += 4 * 32) {   // the keys of four neighbour pairs per lane in flight together
        int pb[4];
        uint64_t ka[4], kb[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + 32 * u;
          pb[u] = -1; ka[u] = kb[u] = 0;
          if (i < n) { pb[u] = a[i]; ka[u] = f.pt_key[a[i - 1]]; kb[u] = f.pt_key[pb[u]]; }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (pb[u] >= 0 && ka[u] != kb[u]) { f.cast_flag[pb[u]] = 1; atomicAdd(&f.warp_cnt[pb[u] >> 5], 1); }
      }
      __syncwarp();
      if (f.profile && lane == 0) { dbg_max(f, 8, n); dbg_add(f, 9, n); }
    }
    prof_flush(f, -1);
    solve_barrier(bar, epoch);
    timeline_mark(f, 58);
  }
  // ---- phase 0c: offsets of the cast points (block 0), then compaction in sequence order (= ray rank order)
  if (blockIdx.x == 0) {
    const int n_warps32 = (f.capacity + 31) >> 5;
    const int total = block_scan_array(f.warp_cnt, f.warp_off, n_warps32);
    if (threadIdx.x == 0) cnt->n_cast = total;
  }
  prof_flush(f, -1);
  solve_barrier(bar, epoch);
  timeline_mark(f, 59);
  const int n_cast = ((volatile int*)&cnt->n_cast)[0];
  for (int base = (gtid & ~31); base < n_points; base += gthreads) {
    const int seq = base + lane;
    const bool c = seq < n_points && __ldcg(&f.cast_flag[seq]) != 0;
    const unsigned m = __ballot_sync(0xffffffffu, c);
    if (c) f.cast_seq[__ldcg(&f.warp_off[seq >> 5]) + __popc(m & ((1u << lane) - 1u))] = seq;
  }
  const int sweep_base0 = ((volatile int*)&f.fc->sweep_base)[0];   // sweep ids are monotonic across frames (31 bits: never wraps in practice)
  const bool wrap = false;
  prof_flush(f, -1);
  solve_barrier(bar, epoch);
  timeline_mark(f, tl++);
  // ---- phase 1: ray set-up (first kH0 steps of every ray)
  for (int r0 = (gtid & ~31); r0 < n_cast; r0 += gthreads) fast3_ray_setup(f, r0 + lane, n_cast);
  prof_flush(f, -1);
  solve_barrier(bar, epoch);
  timeline_mark(f, tl++);
  // ---- phase 2: observed-set fixpoint, rank group by rank group
  int sweep = (wrap ? 0 : sweep_base0);
  sweep = (sweep + 4) & ~3;       // counter slot (sweep + 1) & 3 of the first sweep was zeroed by the frame reset
  const int first_sweep = sweep + 1;
  bool failed = false;
  int g_lo = 0, g_size = f.group0 > 0 ? f.group0 : kGroup0;
  while (g_lo < n_cast && !failed) {
    const int g_hi = (g_lo + g_size < n_cast) ? g_lo + g_size : n_cast;
    bool converged = false;
    for (int it = 0; it < max_sweeps; ++it) {
      ++sweep;
      fast3_sweep(f, sweep, g_lo, g_hi, (WarpDdaScratch*)(s_sort + (threadIdx.x >> 5) * kSortPerWarp));
      prof_flush(f, sweep - first_sweep);
      solve_barrier(bar, epoch);
      if (tl < kTimelineSlots - 12) timeline_mark(f, tl++);
      const int changed = ((volatile int*)cnt->changed)[sweep & 3];
      const int err = ((volatile int*)&cnt->err)[0];
      if (err) { failed = true; break; }
      if (!changed) { converged = true; break; }
    }
    if (!converged) failed = true;
    g_lo = g_hi;
    g_size = (g_size < (1 << 28)) ? g_size * (f.group_mul > 1 ? f.group_mul : 4) : g_size;
  }
  if (gtid == 0) {
    cnt->last_sweep = sweep;
    f.fc->sweep_base = sweep;
    f.fc->sweeps_last = sweep - first_sweep + 1;
    if (failed && !((volatile int*)&cnt->err)[0]) set_err(cnt, 2 /*KSG_ERR_CUDA: the solver did not converge*/);
    if (f.profile) f.fc->timeline[kTimelineSlots - 1] = tl;
  }
  tl = kTimelineSlots - 12;
  timeline_mark(f, tl++);
  // ---- phase 3: table commit + block allocation + records per tile
  if (!failed) fast3_walk_performed<1>(f, n_cast, 0);
  prof_flush(f, -1);
  solve_barrier(bar, epoch);
  timeline_mark(f, tl++);
  timeline_mark(f, tl++);     // (slot kept for the layout of k_fast_solve: there the per-tile count is a phase of its own)
  const bool ok = ((volatile int*)&cnt->err)[0] == 0 && !failed;
  const int n_new_all = ((volatile int*)&cnt->n_new_blocks)[0];
  const int n_new = n_new_all < f.map.new_cap ? n_new_all : f.map.new_cap;
  const int pool_base = ((volatile int*)&cnt->pool_count)[0];
  // ---- phase 4: key segment per tile, updated() bookkeeping, ownership (spatial sharding), new blocks
  const int n_tiles = (int)min((long long)((volatile int*)&f.fc->n_tile_list)[0], f.tile_cap);
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
      if (off + n > f.rec_cap) { set_err(cnt, 4); n = 0; }
      f.tile_list[idx].n = owned ? n : -n;
      f.tile_list[idx].off = off;
    }
  }
  if (ok) fast_block_init(f, n_new, pool_base);
  prof_flush(f, -1);
  solve_barrier(bar, epoch);
  timeline_mark(f, tl++);
  // ---- phase 5: keys into the tile segments (the per-tile counters run back to zero: nothing to clear for the next frame)
  const bool ok2 = ((volatile int*)&cnt->err)[0] == 0 && !failed;
  if (!failed) fast3_walk_performed<2>(f, n_cast, ok2 ? n_tiles : 0);
  if (gtid == 0) {
    int add = n_new;
    if (pool_base + add > f.map.max_blocks) add = f.map.max_blocks - pool_base;
    if (ok) cnt->pool_count = pool_base + (add > 0 ? add : 0);
    cnt->n_tiles = ok2 ? n_tiles : 0;
    cnt->n_records = ((volatile unsigned long long*)&f.fc->rec_cursor)[0];
    f.fc->tile_cursor = 0;
    f.fc->n_tile_list = 0;
    f.fc->rec_cursor = 0;
    if (f.profile) f.prof[0] = f.fc->ovf_count;
    f.fc->ovf_count = 0;
    if (f.profile) { f.fc->dbg[10] = n_mixed; f.fc->dbg[11] = n_cast; }
    f.fc->n_mixed = 0;
    f.fc->m_cursor = 0;
    f.fc->log_count = 0;
  }
  timeline_mark(f, tl++);
}

}  // namespace ksg
