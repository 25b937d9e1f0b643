// collide.cu — K2/K3: MultirotorSimulator::handleCollisions (SIM:295-359) as a uniform-grid spatial
// hash over the packed positions of this shard and of the halo of remote UAVs around it, queried for
// this shard's UAVs only.
//
// The reference rebuilds a nanoflann KD-tree every tick and runs one radius query per UAV with
// squared "radius" 3.0 (SIM:309-328).  Here, per pass:
//   K2a  box      (sharded runs only) bounding box of this shard's positions; a remote UAV further
//                 than `reach` outside it cannot be a neighbour of any local UAV and is not
//                 inserted, so the table holds n_local + halo entries instead of n_global.
//                 Pull exchange (peers mapped over CUDA IPC): remote positions are not copied to
//                 this GPU at all.  Every rank keeps one bounding box per 32 consecutive UAVs next to
//                 its positions (written by the stepping kernel); `count_halo` reads the peers' boxes
//                 over NVLink, skips the groups that cannot reach this shard's box and fetches only
//                 the positions of the others (a halo of a few thousand UAVs instead of the swarm).
//   K2b  count    cell = floor(p / 4 m); bucket = (mix(cy,cz) + cx) mod B, B = 2^bits >= 2 n_global;
//                 rank = atomicAdd(count[bucket], 1).  Cells adjacent in x land in adjacent buckets,
//                 so one stencil row is ONE contiguous range of the grouped records.
//   K2c  scan     begin = exclusive prefix sum of count: one single-pass kernel (decoupled look-back
//                 over 4096-item tiles, tickets handed out in scheduling order).
//   K2d  scatter  rec[begin[bucket] + rank] = {x, y, z, index}  (32-byte records: a candidate costs
//                 exactly one DRAM sector).  This is a counting sort: no radix passes.
//                 Bucket B mirrors bucket 0, so a row never straddles the end of the table.
//   K3   collide  one thread per record; the search ball of radius sqrt(3) < 2 m around p touches at
//                 most 2 cells per axis (interval [p-2, p+2] has the length of one 4 m cell), i.e.
//                 <= 4 stencil rows (cy0..cy1 x cz0..cz1), each one contiguous range cx0..cx1; per
//                 candidate the EXACT reference predicate, evaluated with explicit round-to-nearest
//                 multiplies and adds (no FMA contraction) in nanoflann's order
//                 d2 = ((dx*dx) + dy*dy) + dz*dz, dx = q - p (NF:479-484), accepted iff d2 < 3.0
//                 (NF:305-309, strict) and j != i (SIM:335) and
//                 d2 < ((arm_i+prop_i)+arm_j)+prop_j (SIM:342,346: squared metres against metres —
//                 reproduced as is).
// Bucket aliasing (two cells sharing a bucket) only adds candidates, which fail d2 < 3.0 unless they
// are true neighbours; a true neighbour is accepted only in the probe whose (cy,cz) row is its own
// cell row, so nothing is counted twice.  The arrival order inside a bucket is not deterministic;
// results are: pair lists are sorted on retrieval, and force sums of >= 3 terms are re-accumulated
// in ascending j (sums of <= 2 terms are order-independent bit for bit).
//
// Neighbour lists (single-shard handles).  A UAV moves centimetres per tick, so the table is not
// rebuilt every tick: a rebuild also records, for every UAV, the indices of all UAVs within
// R_list = sqrt(3) + skin of it (<= NL_CAP of them, slot-major [slot][uav]).  The stepping kernel
// reports the largest displacement of any UAV per launch (DevState::disp_max); `decide_kernel` sums
// these bounds into D and the lists stay valid while 2 D <= skin (two UAVs now closer than sqrt(3)
// were closer than sqrt(3) + 2 D when the lists were built).  On such ticks the pass is ONE kernel
// (`check_kernel`: the exact predicate on the current positions of the listed candidates); the
// rebuild (count/scan/scatter/build) sits in the body of a CUDA-graph conditional IF node whose
// condition `decide_kernel` sets on the device, so no host round trip is involved.  Results are the
// same bits either way: the lists only choose which pairs are tested.  Anything that moves UAVs
// other than one stepping launch (set_state, publish_positions, several launches between passes)
// forces a rebuild: the host raises the displacement word to "unbounded" before that pass.  A UAV with more than NL_CAP candidates keeps no list: it remembers where its
// record sits in the (now ageing) table and, every pass, walks the stencil of its build-time cell —
// the records there are a superset of its possible neighbours for as long as the lists are valid —
// testing each candidate's CURRENT position (`check_crowded`).  Only the crowded UAVs pay for that.  Sharded handles use the lists when the peer
// hand-shake carries every rank's displacement bound (pull exchange, api.cu), the full pass otherwise.
// The rebuild's list kernel works with FOUR LANES PER UAV, one per stencil row: each lane walks the
// (short) record range of its row, the four lanes of a UAV agree on list slots through a ballot, and
// the UAVs that have anything to check (a candidate, or the crowded mark) are appended to
// `nl_active` in index order (a second run of the single-pass prefix sum, over "has work" flags): a
// list-only pass runs over those only — typically a third of the swarm — with every lane busy.
// Bit 31 of a UAV's list-count word says "its external force may be non-zero": a pass must REPLACE every
// UAV's force (SIM:356-358), but writing 24 zero bytes over 24 zero bytes for the (vast) majority without a
// neighbour is most of a list-only pass — a UAV with an empty list and a clear bit is left alone.  Whoever
// writes forces elsewhere (mrsb_apply_force, mrsb_forces_written) makes the next pass write them all.
//
// Crash mode (SIM:347-348) marks the NEIGHBOUR crashed.  A shard must not write remote state, so the
// owner of i evaluates the mirrored test d2 < ((arm_j+prop_j)+arm_i)+prop_i — the exact threshold
// the owner of j uses for the directed pair (j,i) — and marks i itself.
#include <algorithm>

#include "internal.h"

namespace {

#define DEV __device__ __forceinline__

#define NL_LIVE 0x80000000u     // bit 31 of nl_count[]: the UAV's external force may be non-zero
#define NL_CROWDED 0x40000000u  // bit 30: more than MRSB_NL_CAP candidates; nl_items[0][uav] = its record in the table

DEV unsigned long long now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// timeline stamp of the current pass (diagnostics; g.tl is nullptr in normal operation)
DEV void stamp(const DevGrid& g, int slot, unsigned long long value) {
  if (g.tl) g.tl[((g.ctl->n_passes - 1ull) % MRSB_TL_TICKS) * 8 + slot] = value;
}

DEV int cell_of(double v, double inv_cell) {
  // floor(v / cell): one F2I.FLOOR — saturates to INT_MIN / INT_MAX, NaN -> 0.  Monotone in v, and the
  // SAME function files a record (count_kernel) and looks for it, which is all the stencil needs.
  return __double2int_rd(__dmul_rn(v, inv_cell));
}

DEV uint32_t row_hash(int cy, int cz) {
  uint32_t h = uint32_t(cy) * 0x9E3779B1u ^ (uint32_t(cz) * 0x85EBCA77u + 0x165667B1u);
  h ^= h >> 15;
  h *= 0x2C1B3C6Du;
  h ^= h >> 12;
  return h;
}

// order-preserving map double -> uint64 (for atomicMin / atomicMax)
DEV unsigned long long enc(double v) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
DEV double dec(unsigned long long e) {
  const unsigned long long b = (e >> 63) ? (e & 0x7fffffffffffffffull) : ~e;
  return __longlong_as_double((long long)b);
}
// inverse of the stepping kernel's fenc(): order-preserving uint32 code -> float
DEV float fdec(uint32_t e) {
  return __uint_as_float((e >> 31) ? (e & 0x7fffffffu) : ~e);
}

// Loads of what every list-only pass reads again (packed positions, compacted entries and lists) and of the positions the
// table rebuild reads: marked evict-last in L2, so that the stepping launch between two passes, which streams ~700 MB of state
// through the 126 MB L2, does not push them out.
DEV uint64_t keep_policy() {
  uint64_t p;
  asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
DEV double ld_keep(const double* p) {
  double v;
  asm("ld.global.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(keep_policy()));
  return v;
}
DEV double ld_keep_nc(const double* p) {  // read-only for the whole kernel
  double v;
  asm("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(keep_policy()));
  return v;
}
DEV int32_t ld_keep(const int32_t* p) {
  int32_t v;
  asm("ld.global.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(keep_policy()));
  return v;
}
DEV uint2 ld_keep(const uint2* p) {
  uint2 v;
  asm("ld.global.L2::cache_hint.v2.u32 {%0, %1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(keep_policy()));
  return v;
}

// ---- where a UAV's current position and collision geometry live -----------------------------------------
// Always in this handle's own arrays.  In pull-exchange runs the slots of REMOTE UAVs in the local position buffer and geometry
// table are a cache that this rank fills itself: at a table rebuild for the whole halo (count_halo_kernel), on every other pass
// for the same UAVs again (refresh_halo_kernel) — every remote UAV a neighbour list or the table can name is one of them.
DEV int owner_of(const PeerView& pv, int64_t gj) {
  int r = 0;
  while (r + 1 < pv.n_ranks && gj >= pv.begin[r + 1]) r++;
  return r;
}
DEV void load_pos(const DevState& s, int64_t gj, double& x, double& y, double& z) {
  const double* p = s.gpos + 3 * gj;
  x = ld_keep(p), y = ld_keep(p + 1), z = ld_keep(p + 2);
}
struct Geom {
  double arm, prop, mass;
};
DEV Geom load_geom(const DevState& s, int64_t gj) {
  const double* p = s.geom + 4 * gj;
  Geom          g;
  g.arm = p[0], g.prop = p[1], g.mass = p[2];
  return g;
}
// Remote memory is always read with ld.global.cv (fetch again, never from a stale line): the owner rewrites it every tick and the
// only ordering between the two GPUs is the hand-shake of decide_kernel.

// ---- bounding boxes --------------------------------------------------------------------------------
__global__ void box_reset_kernel(unsigned long long* aabb) {
  if (threadIdx.x < 3) aabb[threadIdx.x] = ~0ull;
  if (threadIdx.x >= 3 && threadIdx.x < 6) aabb[threadIdx.x] = 0ull;
}

__global__ void __launch_bounds__(256) box_kernel(const double* __restrict__ gpos, int64_t begin, int64_t n, unsigned long long* aabb) {
  unsigned long long lo[3] = {~0ull, ~0ull, ~0ull}, hi[3] = {0ull, 0ull, 0ull};
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const double* p = gpos + 3 * (begin + i);
#pragma unroll
    for (int c = 0; c < 3; c++) {
      const unsigned long long e = enc(p[c]);
      lo[c]                      = min(lo[c], e);
      hi[c]                      = max(hi[c], e);
    }
  }
#pragma unroll
  for (int c = 0; c < 3; c++) {
    for (int o = 16; o > 0; o >>= 1) {
      lo[c] = min(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
      hi[c] = max(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin(&aabb[c], lo[c]);
      atomicMax(&aabb[3 + c], hi[c]);
    }
  }
}

// Pull exchange: this shard's box from its own per-group boxes (DevState::gbox: float codes rounded outwards, so the result
// contains the exact box).  After box_reset_kernel; written in the encoding of box_kernel so that both kinds of halo filter read
// the same words.  A NaN code stays NaN ("no bound").
__global__ void __launch_bounds__(256) box_from_groups_kernel(const uint32_t* __restrict__ gbox, int64_t n_groups, unsigned long long* aabb) {
  uint32_t lo[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, hi[3] = {0u, 0u, 0u};
  for (int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; k < n_groups; k += int64_t(gridDim.x) * blockDim.x) {
    const uint2 a = reinterpret_cast<const uint2*>(gbox + 6 * k)[0], b = reinterpret_cast<const uint2*>(gbox + 6 * k)[1], c = reinterpret_cast<const uint2*>(gbox + 6 * k)[2];
    lo[0] = min(lo[0], a.x), lo[1] = min(lo[1], a.y), lo[2] = min(lo[2], b.x);
    hi[0] = max(hi[0], b.y), hi[1] = max(hi[1], c.x), hi[2] = max(hi[2], c.y);
  }
#pragma unroll
  for (int c = 0; c < 3; c++) {
    lo[c] = __reduce_min_sync(0xffffffffu, lo[c]);
    hi[c] = __reduce_max_sync(0xffffffffu, hi[c]);
    if ((threadIdx.x & 31) == 0) {
      if (lo[c] != 0xFFFFFFFFu) atomicMin(&aabb[c], enc(double(fdec(lo[c]))));
      if (hi[c] != 0u) atomicMax(&aabb[3 + c], enc(double(fdec(hi[c]))));
    }
  }
}

// ---- table build: count, scan, scatter ---------------------------------------------------------------
DEV uint32_t bucket_of(double x, double y, double z, double inv_cell, uint32_t mask) {
  return (row_hash(cell_of(y, inv_cell), cell_of(z, inv_cell)) + uint32_t(cell_of(x, inv_cell))) & mask;
}
// remote: can it reach this shard's box?  (NaN compares false -> kept)
DEV bool outside_box(const unsigned long long* __restrict__ aabb, double reach, double x, double y, double z) {
  return x < dec(aabb[0]) - reach || y < dec(aabb[1]) - reach || z < dec(aabb[2]) - reach || x > dec(aabb[3]) + reach || y > dec(aabb[4]) + reach ||
         z > dec(aabb[5]) + reach;
}

// UAVs [j0, j0 + cnt) of the packed buffer; with `filter`, the ones outside [shard_begin, shard_begin + n_local) only if they can reach the box
__global__ void __launch_bounds__(256) count_kernel(const double* __restrict__ gpos, int64_t j0, int64_t cnt, int64_t shard_begin, int64_t n_local, int filter,
                                                    const unsigned long long* __restrict__ aabb, uint32_t mask, double inv_cell, double reach,
                                                    uint32_t* __restrict__ count, uint32_t* __restrict__ bucket, uint32_t* __restrict__ rank) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= cnt) return;
  const int64_t j = j0 + k;
  const double* p = gpos + 3 * j;
  const double  x = ld_keep_nc(p), y = ld_keep_nc(p + 1), z = ld_keep_nc(p + 2);
  if (filter) {
    const int64_t l = j - shard_begin;
    if ((l < 0 || l >= n_local) && outside_box(aabb, reach, x, y, z)) {
      bucket[j] = 0xFFFFFFFFu;
      return;
    }
  }
  const uint32_t b = bucket_of(x, y, z, inv_cell, mask);
  bucket[j]        = b;
  rank[j]          = atomicAdd(&count[b], 1u);
  // buckets B and B+1 (B = mask+1) mirror buckets 0 and 1 (same records, same ranks), so that the
  // x-adjacent cells of a stencil row are ALWAYS adjacent buckets, also across the end of the table
  if (b <= 1u) atomicAdd(&count[mask + 1u + b], 1u);
}

// Pull exchange: the remote UAVs that can reach this shard's box, fetched from their owners over NVLink — in as few and as
// large requests as possible, and with as many of them in flight as possible (small remote reads are limited by the number a
// single SM can keep outstanding, not by bandwidth).  Two kernels:
//  (1) halo_groups_kernel: a warp takes 16 of a peer's 32-UAV groups at a time — their 16 bounding boxes are 96 consecutive
//      words = three coalesced loads — and lane g < 16 judges group g; groups that come within `reach` of this shard's box go to
//      a work list.
//  (2) halo_fetch_kernel: one warp per listed group: its positions are 96 consecutive doubles = three coalesced loads
//      (redistributed to one UAV per lane by shuffles), its geometry 128 consecutive doubles; every UAV is then filtered on its
//      own, and the kept ones go to the halo list with their bucket, and their position and geometry into the local cache slots.
__global__ void __launch_bounds__(256) halo_groups_kernel(DevGrid g, PeerView pv) {
  const uint32_t full   = 0xffffffffu;
  const int      lane   = threadIdx.x & 31;
  const int64_t  warp   = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t  n_warp = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const double   lo0 = dec(g.aabb[0]) - g.reach, lo1 = dec(g.aabb[1]) - g.reach, lo2 = dec(g.aabb[2]) - g.reach;
  const double   hi0 = dec(g.aabb[3]) + g.reach, hi1 = dec(g.aabb[4]) + g.reach, hi2 = dec(g.aabb[5]) + g.reach;
  // every (peer, chunk of 16 groups) is one work item; items are dealt to the warps round-robin
  int64_t item0 = 0;
  for (int r = 0; r < pv.n_ranks; r++) {
    if (r == pv.rank) continue;
    const int64_t cnt   = pv.begin[r + 1] - pv.begin[r];
    const int64_t n_grp = (cnt + 31) >> 5, n_words = 6 * n_grp, n_chunk = (n_grp + 15) >> 4;
    int64_t       chunk = (warp - item0 % n_warp + n_warp) % n_warp;  // the first chunk of this peer that falls to this warp
    item0 += n_chunk;
    for (; chunk < n_chunk; chunk += n_warp) {
      uint32_t w[3];
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const int64_t k = chunk * 96 + 32 * c + lane;
        w[c]            = k < n_words ? __ldcv(pv.box[r] + k) : 0u;
      }
      auto word = [&](int k) {  // word k (0..95) of the chunk: register k / 32 of lane k % 32
        const uint32_t a = __shfl_sync(full, w[0], k & 31), b = __shfl_sync(full, w[1], k & 31), c = __shfl_sync(full, w[2], k & 31);
        return k < 32 ? a : (k < 64 ? b : c);
      };
      const int    k0 = 6 * (lane & 15);
      const double b0 = fdec(word(k0)), b1 = fdec(word(k0 + 1)), b2 = fdec(word(k0 + 2));
      const double t0 = fdec(word(k0 + 3)), t1 = fdec(word(k0 + 4)), t2 = fdec(word(k0 + 5));
      const bool   reach = lane < 16 && chunk * 16 + lane < n_grp && !(b0 > hi0 || b1 > hi1 || b2 > hi2 || t0 < lo0 || t1 < lo1 || t2 < lo2);  // NaN bounds: kept
      const uint32_t todo = __ballot_sync(full, reach);
      if (todo) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(g.halo_work_n, uint32_t(__popc(todo)));
        base = __shfl_sync(full, base, 0);
        if (reach) g.halo_work[base + __popc(todo & ((1u << lane) - 1u))] = (uint32_t(r) << 26) | uint32_t(chunk * 16 + lane);
      }
    }
  }
}

__global__ void __launch_bounds__(256) halo_fetch_kernel(DevState s, DevGrid g, PeerView pv, uint32_t mask) {
  const uint32_t full   = 0xffffffffu;
  const int      lane   = threadIdx.x & 31;
  const int64_t  warp   = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t  n_warp = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const int64_t  n_work = *g.halo_work_n;
  const double   lo0 = dec(g.aabb[0]) - g.reach, lo1 = dec(g.aabb[1]) - g.reach, lo2 = dec(g.aabb[2]) - g.reach;
  const double   hi0 = dec(g.aabb[3]) + g.reach, hi1 = dec(g.aabb[4]) + g.reach, hi2 = dec(g.aabb[5]) + g.reach;
  for (int64_t item = warp; item < n_work; item += n_warp) {
    const uint32_t code  = g.halo_work[item];
    const int      r     = int(code >> 26);
    const int64_t  grp   = code & 0x3FFFFFFu;
    const int64_t  first = pv.begin[r], cnt = pv.begin[r + 1] - first;
    const int64_t  l0    = 32 * grp;
    const int64_t  n_uav = min(int64_t(32), cnt - l0);
    const double*  base  = pv.pos[r] + 3 * (first + l0);
    const double2* gbase = reinterpret_cast<const double2*>(pv.geom[r] + 4 * (first + l0));
    // every remote load of the group first (positions: 3 coalesced rows; geometry: this lane's UAV): one NVLink round trip
    double d[3];
#pragma unroll
    for (int c = 0; c < 3; c++) d[c] = 32 * c + lane < 3 * n_uav ? __ldcv(base + 32 * c + lane) : 0.0;
    double2 ga = make_double2(0.0, 0.0), gb = ga;
    if (lane < n_uav) {
      ga = __ldcv(gbase + 2 * lane);
      gb = __ldcv(gbase + 2 * lane + 1);
    }
    auto pick = [&](int k) {
      const double a = __shfl_sync(full, d[0], k & 31), b = __shfl_sync(full, d[1], k & 31), c = __shfl_sync(full, d[2], k & 31);
      return k < 32 ? a : (k < 64 ? b : c);
    };
    const double x = pick(3 * lane), y = pick(3 * lane + 1), z = pick(3 * lane + 2);
    if (lane >= n_uav) continue;
    if (x < lo0 || y < lo1 || z < lo2 || x > hi0 || y > hi1 || z > hi2) continue;
    const int64_t  gj = first + l0 + lane;
    const uint32_t bk = bucket_of(x, y, z, g.inv_cell, mask);
    const uint32_t rk = atomicAdd(&g.count[bk], 1u);
    if (bk <= 1u) atomicAdd(&g.count[mask + 1u + bk], 1u);
    const uint32_t slot = atomicAdd(g.halo_n, 1u);
    if (int64_t(slot) < g.halo_cap) {
      g.halo_rec[slot]    = make_double4(x, y, z, __longlong_as_double((long long)gj));
      g.halo_bucket[slot] = bk;
      g.halo_rank[slot]   = rk;
    }
    double* lp = s.gpos + 3 * gj;
    lp[0] = x, lp[1] = y, lp[2] = z;
    double2* lg = reinterpret_cast<double2*>(s.geom + 4 * gj);
    lg[0] = ga, lg[1] = gb;
  }
}

// Pull exchange, passes between rebuilds: the CURRENT positions (and geometry) of the halo UAVs of the last rebuild, from their
// owners into the local cache slots.  A few thousand UAVs; small CTAs so that the remote reads spread over all SMs.
__global__ void __launch_bounds__(64) refresh_halo_kernel(DevState s, DevGrid g, PeerView pv) {
  if (blockIdx.x == 0 && threadIdx.x == 0) stamp(g, 3, now_ns());
  if (g.ctl->rebuild) return;  // this pass rebuilds: count_halo_kernel fetches the (new) halo
  const int64_t n = min(int64_t(*g.halo_n), g.halo_cap);
  for (int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; k < n; k += int64_t(gridDim.x) * blockDim.x) {
    const int64_t  gj = __double_as_longlong(g.halo_rec[k].w);
    const int      r  = owner_of(pv, gj);
    const double*  p  = pv.pos[r] + 3 * gj;
    const double2* gp = reinterpret_cast<const double2*>(pv.geom[r] + 4 * gj);
    // all five remote loads first: one NVLink round trip
    const double  x = __ldcv(p), y = __ldcv(p + 1), z = __ldcv(p + 2);
    const double2 a = __ldcv(gp), b = __ldcv(gp + 1);
    double*       lp = s.gpos + 3 * gj;
    lp[0] = x, lp[1] = y, lp[2] = z;
    double2* lg = reinterpret_cast<double2*>(s.geom + 4 * gj);
    lg[0] = a, lg[1] = b;
  }
}

// Exclusive prefix sum of `in` in ONE pass: tiles of 4096 items, tile numbers taken from a ticket counter (so a tile only ever
// waits for tiles that are already running), per-tile status word {2-bit flag | 32-bit value}: A = the tile's own sum, P = the
// inclusive prefix up to and including the tile; a warp looks back over 32 predecessors at a time.  state[0] = ticket counter,
// state[1 + t] = status of tile t, all zero before the launch.
#define SCAN_PER_THREAD 16
#define SCAN_TILE (256 * SCAN_PER_THREAD)
#define SCAN_FLAG_A (1ull << 32)
#define SCAN_FLAG_P (2ull << 32)
// HASWORK: the items are neighbour-list count words and the value summed is "has something to check" (0 / 1) — the exclusive sum
// is then the UAV's slot in the compacted list `nl_active` (index order).
template <bool HASWORK>
__global__ void __launch_bounds__(256) scan_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int64_t n, unsigned long long* state) {
  __shared__ uint32_t s_tile, s_warp[8], s_prefix;
  const uint32_t      full = 0xffffffffu;
  const int           lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_tile = uint32_t(atomicAdd(&state[0], 1ull));
  __syncthreads();
  const int64_t tile = s_tile;
  const int64_t base = tile * SCAN_TILE + int64_t(threadIdx.x) * SCAN_PER_THREAD;
  uint32_t      v[SCAN_PER_THREAD];
  if (base + SCAN_PER_THREAD <= n) {
#pragma unroll
    for (int q = 0; q < SCAN_PER_THREAD / 4; q++) {
      const uint4 a = reinterpret_cast<const uint4*>(in + base)[q];
      v[4 * q] = a.x, v[4 * q + 1] = a.y, v[4 * q + 2] = a.z, v[4 * q + 3] = a.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < SCAN_PER_THREAD; k++) v[k] = base + k < n ? in[base + k] : 0u;
  }
  if (HASWORK) {
#pragma unroll
    for (int k = 0; k < SCAN_PER_THREAD; k++) v[k] = (v[k] & 0x7FFFFFFFu) != 0u ? 1u : 0u;  // everything but the NL_LIVE bit: candidates or the crowded mark
  }
  uint32_t mine = 0;
#pragma unroll
  for (int k = 0; k < SCAN_PER_THREAD; k++) mine += v[k];
  uint32_t incl = mine;  // inclusive scan of the thread sums inside the warp
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(full, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  uint32_t warp_off = 0, total = 0;
#pragma unroll
  for (int w = 0; w < 8; w++) {
    if (w < wid) warp_off += s_warp[w];
    total += s_warp[w];
  }
  if (wid == 0) {
    volatile unsigned long long* st = state + 1;
    uint32_t                     prefix = 0;
    if (tile == 0) {
      if (lane == 0) st[0] = SCAN_FLAG_P | total;
    } else {
      if (lane == 0) st[tile] = SCAN_FLAG_A | total;
      int64_t look = tile - 1;
      while (true) {
        const int64_t      t = look - lane;
        unsigned long long w = t >= 0 ? st[t] : SCAN_FLAG_P;  // before tile 0: inclusive prefix 0
        while (__any_sync(full, (w >> 32) == 0ull)) {
          if ((w >> 32) == 0ull) w = st[t];
        }
        const uint32_t pm    = __ballot_sync(full, (w >> 32) == 2ull);
        const int      first = pm ? __ffs(int(pm)) - 1 : 32;
        uint32_t       add   = lane <= first ? uint32_t(w) : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) add += __shfl_xor_sync(full, add, o);
        prefix += add;
        if (pm) break;
        look -= 32;
      }
      if (lane == 0) st[tile] = SCAN_FLAG_P | (unsigned long long)(prefix + total);
    }
    if (lane == 0) s_prefix = prefix;
  }
  __syncthreads();
  uint32_t run = s_prefix + warp_off + (incl - mine);
  if (base + SCAN_PER_THREAD <= n) {
#pragma unroll
    for (int q = 0; q < SCAN_PER_THREAD / 4; q++) {
      uint4 a;
      a.x = run, run += v[4 * q];
      a.y = run, run += v[4 * q + 1];
      a.z = run, run += v[4 * q + 2];
      a.w = run, run += v[4 * q + 3];
      reinterpret_cast<uint4*>(out + base)[q] = a;
    }
  } else {
#pragma unroll
    for (int k = 0; k < SCAN_PER_THREAD; k++) {
      if (base + k < n) out[base + k] = run;
      run += v[k];
    }
  }
}

__global__ void __launch_bounds__(256) scatter_kernel(const double* __restrict__ gpos, int64_t j0, int64_t cnt, const uint32_t* __restrict__ bucket,
                                                      const uint32_t* __restrict__ rank, const uint32_t* __restrict__ begin, uint32_t n_buckets,
                                                      double4* __restrict__ rec) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= cnt) return;
  const int64_t  j = j0 + k;
  const uint32_t b = bucket[j];
  if (b == 0xFFFFFFFFu) return;
  const double*  q = gpos + 3 * j;
  const double4  r = make_double4(ld_keep_nc(q), ld_keep_nc(q + 1), ld_keep_nc(q + 2), __longlong_as_double((long long)j));
  const uint32_t t = rank[j];
  rec[begin[b] + t] = r;
  if (b <= 1u) rec[begin[n_buckets + b] + t] = r;  // mirrors of buckets 0 and 1
}

__global__ void __launch_bounds__(256) scatter_halo_kernel(DevGrid g) {
  const int64_t n = min(int64_t(*g.halo_n), g.halo_cap);
  for (int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; k < n; k += int64_t(gridDim.x) * blockDim.x) {
    const double4  r = g.halo_rec[k];
    const uint32_t b = g.halo_bucket[k], t = g.halo_rank[k];
    g.rec[g.begin[b] + t] = r;
    if (b <= 1u) g.rec[g.begin[g.n_buckets + b] + t] = r;
  }
}

// nanoflann L2 metric for dim 3, no contraction
DEV double nf_dist2(double ax, double ay, double az, double bx, double by, double bz) {
  const double d0 = __dsub_rn(ax, bx), d1 = __dsub_rn(ay, by), d2 = __dsub_rn(az, bz);
  double       r  = __dmul_rn(d0, d0);
  r               = __dadd_rn(r, __dmul_rn(d1, d1));
  r               = __dadd_rn(r, __dmul_rn(d2, d2));
  return r;
}

// The <= 4 stencil rows around q.  The search ball (radius < reach = cell / 2) fits into two cells
// per axis: {c0, c0 + 1} with c0 = cell_of(q - reach) — for any p with |p - q| < r_search,
// q - reach <= p < (q - reach) + cell, and cell_of is monotone.  Each row (cy, cz) is ONE record
// range: buckets b0, b0 + 1 with b0 = bucket of (cx0, cy, cz).
struct Stencil {
  int      rcy[4], rcz[4];
  uint32_t lo[4], hi[4];
};
DEV Stencil stencil_of(const DevGrid& g, double qx, double qy, double qz) {
  Stencil        st;
  const uint32_t mask = g.n_buckets - 1;
  const int      cx0 = cell_of(qx - g.reach, g.inv_cell), cy0 = cell_of(qy - g.reach, g.inv_cell), cz0 = cell_of(qz - g.reach, g.inv_cell);
#pragma unroll
  for (int k = 0; k < 4; k++) {
    st.rcy[k]         = cy0 + (k & 1);
    st.rcz[k]         = cz0 + ((k >> 1) & 1);
    const uint32_t b0 = (row_hash(st.rcy[k], st.rcz[k]) + uint32_t(cx0)) & mask;
    st.lo[k]          = g.begin[b0];
    st.hi[k]          = g.begin[b0 + 2];  // b0 + 2 <= mask + 2: begin[] has the two mirror buckets and a sentinel
  }
  return st;
}

// One accepted candidate (d2 < 3.0 already established): SIM:342-353 for the directed pair (i, j).
struct PairAcc {
  double fx = 0.0, fy = 0.0, fz = 0.0;
  bool   crashed_me = false;
};
DEV void process_pair(const DevState& s, const DevGrid& g, int crash_mode, double rebounce, int64_t gi, double qx, double qy, double qz, const Geom& Gi,
                      int64_t gj, double rx_, double ry_, double rz_, PairAcc& acc) {
  const double ai = Gi.arm, pi_ = Gi.prop, mi = Gi.mass;
  const double api = __dadd_rn(ai, pi_);
  const double d2  = nf_dist2(qx, qy, qz, rx_, ry_, rz_);
  const Geom   Gj  = load_geom(s, gj);
  const double aj = Gj.arm, pj = Gj.prop;
  const double crit_ij = __dadd_rn(__dadd_rn(api, aj), pj);  // SIM:342
  if (d2 < crit_ij) {                                         // SIM:346
    const unsigned long long slot = atomicAdd(g.counters, 1ull);
    if (slot < (unsigned long long)g.pair_cap) {
      g.pairs[2 * slot]     = int32_t(gi);
      g.pairs[2 * slot + 1] = int32_t(gj);
    }
    if (!crash_mode) {
      // rebounce * normalized(x_i - x_j) * m_i * (m_j / (m_i + m_j))   (SIM:350), Eigen evaluation order
      const double rx = __dsub_rn(qx, rx_), ry = __dsub_rn(qy, ry_), rz = __dsub_rn(qz, rz_);
      const double z  = __dadd_rn(__dmul_rn(rx, rx), __dadd_rn(__dmul_rn(ry, ry), __dmul_rn(rz, rz)));
      double       nx = rx, ny = ry, nz = rz;
      if (z > 0.0) {
        const double sq = __dsqrt_rn(z);
        nx              = __ddiv_rn(rx, sq);
        ny              = __ddiv_rn(ry, sq);
        nz              = __ddiv_rn(rz, sq);
      }
      const double mj = Gj.mass;
      const double wt = __ddiv_rn(mj, __dadd_rn(mi, mj));
      acc.fx          = __dadd_rn(acc.fx, __dmul_rn(__dmul_rn(__dmul_rn(rebounce, nx), mi), wt));
      acc.fy          = __dadd_rn(acc.fy, __dmul_rn(__dmul_rn(__dmul_rn(rebounce, ny), mi), wt));
      acc.fz          = __dadd_rn(acc.fz, __dmul_rn(__dmul_rn(__dmul_rn(rebounce, nz), mi), wt));
    }
  }
  if (crash_mode) {
    const double crit_ji = __dadd_rn(__dadd_rn(__dadd_rn(aj, pj), ai), pi_);  // threshold of the directed pair (j,i)
    if (d2 < crit_ji) acc.crashed_me = true;
  }
}

// SIM:356-358: forces replace external_force_ for the next tick (zero in crash mode, SIM:315-319)
// li: (external) local index; the force rows and the flags live in the UAV's slot of the tiled arrays (DevState::perm)
DEV int64_t slot_of(const DevState& s, int64_t li) { return s.perm ? int64_t(s.perm[li]) : li; }
DEV void store_result(const DevState& s, int64_t li, const PairAcc& acc) {
  const int64_t sl = slot_of(s, li);
  s.fext[tix(F3_ROWS, 0, sl)] = acc.fx;
  s.fext[tix(F3_ROWS, 1, sl)] = acc.fy;
  s.fext[tix(F3_ROWS, 2, sl)] = acc.fz;
  if (acc.crashed_me) s.flags[sl] |= FLAG_CRASHED;
}
DEV bool nonzero(const PairAcc& acc) {
  return !(acc.fx == 0.0 && acc.fy == 0.0 && acc.fz == 0.0);  // NaN counts as non-zero
}

#ifndef MRSB_COLLIDE_MINB
#define MRSB_COLLIDE_MINB 7  // 71 registers, no spills; 8 and 10 (64 / 48 registers) measured no faster
#endif
// The full pass: every record against its stencil (handles without neighbour lists).
__global__ void __launch_bounds__(128, MRSB_COLLIDE_MINB) collide_kernel(DevState s, DevGrid g, int crash_mode, double rebounce) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= int64_t(g.begin[g.n_buckets])) return;  // beyond the primary records (the mirror buckets hold copies)
  const double4 q  = g.rec[p];
  const int64_t gi = __double_as_longlong(q.w);
  const int64_t li = gi - s.shard_begin;
  if (li < 0 || li >= s.n) return;  // halo record: its owner handles it

  const Stencil st = stencil_of(g, q.x, q.y, q.z);
  double4       first[4];
#pragma unroll
  for (int k = 0; k < 4; k++) first[k] = st.lo[k] < st.hi[k] ? g.rec[st.lo[k]] : q;  // the four leading candidates are fetched together

  // ---- phase 1 (cheap, unrolled): which records are in the search ball?  A record r found in row k
  // is a genuine, not-yet-seen neighbour iff d2 < 3.0 AND its own cell row is row k (rejects bucket
  // aliases and duplicates).  Almost every UAV has none; keep the first two, count the rest.
  auto in_ball = [&](const double4& r, int k) {
    if (__double_as_longlong(r.w) == gi) return false;  // SIM:335
    const double d2 = nf_dist2(q.x, q.y, q.z, r.x, r.y, r.z);
    if (!(d2 < 3.0)) return false;  // NF:305-309
    return cell_of(r.y, g.inv_cell) == st.rcy[k] && cell_of(r.z, g.inv_cell) == st.rcz[k];
  };
  int      n_ball = 0;
  uint32_t h0 = 0, h1 = 0;
  auto     note = [&](uint32_t t) {
    if (n_ball == 0) h0 = t;
    if (n_ball == 1) h1 = t;
    n_ball++;
  };
#pragma unroll
  for (int k = 0; k < 4; k++) {
    if (st.lo[k] < st.hi[k]) {
      if (in_ball(first[k], k)) note(st.lo[k]);
      for (uint32_t t = st.lo[k] + 1; t < st.hi[k]; t++)
        if (in_ball(g.rec[t], k)) note(t);
    }
  }

  PairAcc acc;
  if (n_ball > 0) {
    // ---- phase 2 (rare, one copy of the heavy code): thresholds, pair list, force, crash flag
    const Geom Gi      = load_geom(s, gi);
    auto       process = [&](const double4& r) { process_pair(s, g, crash_mode, rebounce, gi, q.x, q.y, q.z, Gi, __double_as_longlong(r.w), r.x, r.y, r.z, acc); };
    if (n_ball <= 2) {
      // sums of <= 2 terms do not depend on the order
      for (int c = 0; c < n_ball; c++) {
        process(g.rec[h0]);
        h0 = h1;
      }
    } else {
      // >= 3 neighbours in the ball: visit them in ascending j so that the force sum does not
      // depend on the arrival order inside the buckets (selection by repeated scan; rare)
      int64_t last = -1;
      for (int c = 0; c < n_ball; c++) {
        int64_t  best = INT64_MAX;
        uint32_t bt   = 0;
        for (int k = 0; k < 4; k++) {
          for (uint32_t t = st.lo[k]; t < st.hi[k]; t++) {
            const double4 r  = g.rec[t];
            const int64_t gj = __double_as_longlong(r.w);
            if (gj <= last || gj >= best || !in_ball(r, k)) continue;
            best = gj;
            bt   = t;
          }
        }
        if (best == INT64_MAX) break;
        process(g.rec[bt]);
        last = best;
      }
    }
  }
  store_result(s, li, acc);
  if (g.nl_count) g.nl_count[li] = (g.nl_count[li] & ~NL_LIVE) | (nonzero(acc) ? NL_LIVE : 0u);
}

// ---- neighbour lists ---------------------------------------------------------------------------

// FOUR LANES PER RECORD: lane k of a record looks up the record range of stencil row (cy0 + (k & 1), cz0 + (k >> 1)); the four
// ranges' candidates are then dealt to the four lanes round-robin.  Every round each lane tests two candidates; the four lanes of a record learn from one ballot how many of them accept,
// which gives every accepted candidate its list slot without atomics.  A warp handles 8 records, a CTA 32; CTAs stride over the
// table.  Afterwards lane 0 of the record writes the count word.
__global__ void __launch_bounds__(128) build_lists_kernel(DevState s, DevGrid g) {
  if (blockIdx.x == 0 && threadIdx.x == 0) stamp(g, 7, now_ns());
  const uint32_t full  = 0xffffffffu;
  const int      lane  = threadIdx.x & 31;
  const int      k     = threadIdx.x & 3;
  const int64_t  n_rec = int64_t(g.begin[g.n_buckets]);
  const uint32_t quad  = 0xFu << (lane & ~3);            // the four lanes of my record
  const uint32_t below = quad & ((1u << lane) - 1u);     // ... of them, the ones before me
  const uint32_t mask  = g.n_buckets - 1;
  const bool     write_all = g.ctl->n_passes <= g.ctl->write_all_until;
  for (int64_t p0 = int64_t(blockIdx.x) * 32; p0 < n_rec; p0 += int64_t(gridDim.x) * 32) {
    const int64_t p   = p0 + (threadIdx.x >> 2);
    const bool    has = p < n_rec;
    double4       q   = make_double4(0.0, 0.0, 0.0, 0.0);
    if (has) q = g.rec[p];
    const int64_t gi   = __double_as_longlong(q.w);
    const int64_t li   = gi - s.shard_begin;
    const bool    mine = has && li >= 0 && li < s.n;  // halo records are only candidates
    // lane k looks up the record range of stencil row k = (cy0 + (k & 1), cz0 + (k >> 1)); the quad then shares the four ranges and
    // deals their candidates out round-robin, so that every lane has the same amount of work whatever the rows' lengths are
    // (rows of the cell layer above or below the swarm are empty)
    const int cx0 = cell_of(q.x - g.reach, g.inv_cell), cy0 = cell_of(q.y - g.reach, g.inv_cell), cz0 = cell_of(q.z - g.reach, g.inv_cell);
    uint32_t  lo = 0, len = 0;
    if (mine) {
      const uint32_t b0 = (row_hash(cy0 + (k & 1), cz0 + (k >> 1)) + uint32_t(cx0)) & mask;
      lo                = g.begin[b0];
      len               = g.begin[b0 + 2] - lo;
    }
    const int      qb  = lane & ~3;
    const uint32_t lo0 = __shfl_sync(full, lo, qb), lo1 = __shfl_sync(full, lo, qb + 1), lo2 = __shfl_sync(full, lo, qb + 2), lo3 = __shfl_sync(full, lo, qb + 3);
    const uint32_t c1  = __shfl_sync(full, len, qb);
    const uint32_t c2  = c1 + __shfl_sync(full, len, qb + 1);
    const uint32_t c3  = c2 + __shfl_sync(full, len, qb + 2);
    const uint32_t tot = c3 + __shfl_sync(full, len, qb + 3);
    auto where = [&](uint32_t c, int& row) -> uint32_t {  // candidate c of the concatenated ranges: its row and its record index
      row = int(c >= c1) + int(c >= c2) + int(c >= c3);
      return row == 0 ? lo0 + c : (row == 1 ? lo1 + (c - c1) : (row == 2 ? lo2 + (c - c2) : lo3 + (c - c3)));
    };
    uint32_t cnt = 0;
    for (uint32_t c = uint32_t(k); __any_sync(full, c < tot); c += 8) {
      // two candidates per lane and round: both loads first, then the tests
      double4 r[2];
      int     row[2] = {0, 0};
#pragma unroll
      for (int u = 0; u < 2; u++)
        if (c + 4 * u < tot) r[u] = g.rec[where(c + 4 * u, row[u])];
#pragma unroll
      for (int u = 0; u < 2; u++) {
        bool    take = false;
        int32_t gj   = 0;
        if (c + 4 * u < tot) {
          gj = int32_t(__double_as_longlong(r[u].w));
          if (int64_t(gj) != gi && nf_dist2(q.x, q.y, q.z, r[u].x, r[u].y, r[u].z) < g.list_r2 && cell_of(r[u].y, g.inv_cell) == cy0 + (row[u] & 1) &&
              cell_of(r[u].z, g.inv_cell) == cz0 + (row[u] >> 1))  // the last two: not a bucket alias, not seen in another row
            take = true;
        }
        const uint32_t bal = __ballot_sync(full, take) & quad;
        if (take) {
          const uint32_t slot = cnt + __popc(bal & below);
          if (slot < MRSB_NL_CAP) g.nl_items[int64_t(slot) * g.nl_ld + li] = gj;
        }
        cnt += __popc(bal);
      }
    }
    __syncwarp();  // the list stores above are ordered before the stores below
    const bool lead = mine && k == 0;
    if (lead) {
      uint32_t live = g.nl_count[li] & NL_LIVE;
      if (cnt == 0u && (live || write_all)) {
        // nobody within the list radius: this UAV is not visited again until the next rebuild, so its force
        // (left from an earlier collision, or written from outside) is replaced by zero right here (SIM:356-358)
        const int64_t sl            = slot_of(s, li);
        s.fext[tix(F3_ROWS, 0, sl)] = 0.0;
        s.fext[tix(F3_ROWS, 1, sl)] = 0.0;
        s.fext[tix(F3_ROWS, 2, sl)] = 0.0;
        live                        = 0u;
      }
      if (cnt > MRSB_NL_CAP) {
        // too crowded for a list: remember the record instead (check_crowded walks its stencil every pass)
        g.nl_items[li] = int32_t(uint32_t(p));
        g.nl_count[li] = NL_CROWDED | live;
        atomicAdd(&g.ctl->n_crowded, 1u);
      } else {
        g.nl_count[li] = cnt | live;
      }
    }
  }
}

// The UAVs with something to check on list-only passes, compacted in INDEX order (their accesses to the list columns, positions
// and forces then coalesce): slot = exclusive count of such UAVs before it (scan_kernel<true> over the count words).
// The compacted entry holds everything a list-only pass needs to start on: {local index, count word} in `nl_active`, and the
// UAV's list again, slot-major by ENTRY (`act_items`) — the check then has two dependent memory levels (entry -> positions)
// instead of four (entry -> count word -> list -> positions).
__global__ void __launch_bounds__(256) compact_kernel(DevGrid g, const uint32_t* __restrict__ slot, int64_t n) {
  const int64_t li = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (li >= n) return;
  const uint32_t word = g.nl_count[li];
  const bool     work = (word & 0x7FFFFFFFu) != 0u;
  if (work) {
    const uint32_t k   = slot[li];
    g.nl_active[k]     = make_uint2(uint32_t(li), word);
    const uint32_t cnt = (word & NL_CROWDED) ? 1u : (word & ~(NL_LIVE | NL_CROWDED));  // crowded: slot 0 holds its record index
    for (uint32_t c = 0; c < cnt; c++) g.act_items[int64_t(c) * g.nl_ld + k] = g.nl_items[int64_t(c) * g.nl_ld + li];
  }
  if (li == n - 1) g.ctl->n_active = slot[li] + (work ? 1u : 0u);
}

// A UAV without a list: every record of the stencil around its BUILD-TIME position, tested at the
// candidates' CURRENT positions (the table only says who they are).  Same structure as collide_kernel.
DEV void check_crowded(const DevState& s, const DevGrid& g, int crash_mode, double rebounce, int64_t gi, uint32_t rec_index, PairAcc& acc) {
  const double4 qb = g.rec[rec_index];
  const Stencil st = stencil_of(g, qb.x, qb.y, qb.z);
  const double* qp = s.gpos + 3 * gi;
  const double  qx = qp[0], qy = qp[1], qz = qp[2];
  auto in_ball = [&](const double4& r, int k) {  // r: the candidate's record (build-time position: decides the row it was filed under)
    const int64_t gj = __double_as_longlong(r.w);
    if (gj == gi) return false;
    if (cell_of(r.y, g.inv_cell) != st.rcy[k] || cell_of(r.z, g.inv_cell) != st.rcz[k]) return false;  // bucket alias / duplicate
    double rx, ry, rz;
    load_pos(s, gj, rx, ry, rz);
    return nf_dist2(qx, qy, qz, rx, ry, rz) < 3.0;
  };
  const Geom Gi      = load_geom(s, gi);
  auto       process = [&](int64_t gj) {
    double rx, ry, rz;
    load_pos(s, gj, rx, ry, rz);
    process_pair(s, g, crash_mode, rebounce, gi, qx, qy, qz, Gi, gj, rx, ry, rz, acc);
  };
  int     n_ball = 0;
  int64_t h0 = 0, h1 = 0;
  for (int k = 0; k < 4; k++)
    for (uint32_t t = st.lo[k]; t < st.hi[k]; t++) {
      const double4 r = g.rec[t];
      if (!in_ball(r, k)) continue;
      if (n_ball == 0) h0 = __double_as_longlong(r.w);
      if (n_ball == 1) h1 = __double_as_longlong(r.w);
      n_ball++;
    }
  if (n_ball <= 2) {
    if (n_ball >= 1) process(h0);
    if (n_ball == 2) process(h1);
    return;
  }
  int64_t last = -1;  // >= 3: ascending j
  for (int c = 0; c < n_ball; c++) {
    int64_t best = INT64_MAX;
    for (int k = 0; k < 4; k++)
      for (uint32_t t = st.lo[k]; t < st.hi[k]; t++) {
        const double4 r  = g.rec[t];
        const int64_t gj = __double_as_longlong(r.w);
        if (gj <= last || gj >= best || !in_ball(r, k)) continue;
        best = gj;
      }
    if (best == INT64_MAX) break;
    process(best);
    last = best;
  }
}

// One UAV that has something to check: the exact predicate on the CURRENT positions of its listed candidates.
// (Tried and dropped: remembering each candidate's distance at build time and skipping the fetch while
// d_build - 2 D is still above sqrt(3) — the extra dependent load cost more than the skipped gathers.)
// k: the UAV's entry in the compacted arrays; first4: the first four slots of its list (fetched with the entry)
DEV void check_one(const DevState& s, const DevGrid& g, int crash_mode, double rebounce, uint32_t k, int64_t li, uint32_t word, const int32_t* first4) {
  const uint32_t cnt  = word & ~(NL_LIVE | NL_CROWDED);
  // forces were written from outside since the last pass (this pass' index <= write_all_until): replace them all
  const bool     live = (word & NL_LIVE) || g.ctl->n_passes <= g.ctl->write_all_until;
  PairAcc acc;
  if (word & NL_CROWDED) {
    check_crowded(s, g, crash_mode, rebounce, li + s.shard_begin, uint32_t(first4[0]), acc);
  } else if (cnt) {
    const int64_t gi = li + s.shard_begin;
    const double* qp = s.gpos + 3 * gi;
    const double  qx = ld_keep(qp), qy = ld_keep(qp + 1), qz = ld_keep(qp + 2);
    uint32_t      hits = 0;
    for (uint32_t base = 0; base < cnt; base += 4) {
      // four candidates at a time: indices, then positions, then distances (independent loads in flight)
      int32_t gj[4];
      double  r[4][3];
#pragma unroll
      for (int u = 0; u < 4; u++) gj[u] = base + u < cnt ? (base == 0 ? first4[u] : ld_keep(g.act_items + int64_t(base + u) * g.nl_ld + k)) : -1;
#pragma unroll
      for (int u = 0; u < 4; u++) load_pos(s, int64_t(max(gj[u], 0)), r[u][0], r[u][1], r[u][2]);
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (gj[u] >= 0 && nf_dist2(qx, qy, qz, r[u][0], r[u][1], r[u][2]) < 3.0) hits |= 1u << (base + u);  // NF:305-309
    }
    if (hits) {
      const Geom Gi      = load_geom(s, gi);
      auto       process = [&](uint32_t c) {
        const int64_t gj = g.act_items[int64_t(c) * g.nl_ld + k];
        double        rx, ry, rz;
        load_pos(s, gj, rx, ry, rz);
        process_pair(s, g, crash_mode, rebounce, gi, qx, qy, qz, Gi, gj, rx, ry, rz, acc);
      };
      if (__popc(hits) <= 2) {
        // sums of <= 2 terms do not depend on the order
        while (hits) {
          process(uint32_t(__ffs(int(hits)) - 1));
          hits &= hits - 1;
        }
      } else {
        // >= 3: ascending j, like collide_kernel
        int64_t last = -1;
        while (hits) {
          int64_t  best = INT64_MAX;
          uint32_t bc   = 0;
          for (uint32_t m = hits; m; m &= m - 1) {
            const uint32_t c  = uint32_t(__ffs(int(m)) - 1);
            const int64_t  gj = g.act_items[int64_t(c) * g.nl_ld + k];
            if (gj > last && gj < best) best = gj, bc = c;
          }
          if (best == INT64_MAX) break;
          process(bc);
          last = best;
          hits &= ~(1u << bc);
        }
      }
    }
  }
  const bool nz = nonzero(acc);
  if (live || nz) store_result(s, li, acc);
  else if (acc.crashed_me) s.flags[slot_of(s, li)] |= FLAG_CRASHED;
  if (nz != bool(word & NL_LIVE)) {
    const uint32_t nw = (word & ~NL_LIVE) | (nz ? NL_LIVE : 0u);
    g.nl_count[li]    = nw;
    g.nl_active[k].y  = nw;
  }
}

// A list-only pass: the compacted UAVs that have something to check, grid-stride.
// skip_if_rebuild: this launch runs BESIDE the conditional rebuild node of the graph, not behind it; on a rebuilding pass it does
// nothing — the rebuild's body ends with its own launch of this kernel.
#ifndef MRSB_CHECK_THREADS
#define MRSB_CHECK_THREADS 256
#define MRSB_CHECK_MINB 4
#endif
__global__ void __launch_bounds__(MRSB_CHECK_THREADS, MRSB_CHECK_MINB) check_kernel(DevState s, DevGrid g, int crash_mode, double rebounce, int skip_if_rebuild) {
  if (skip_if_rebuild && g.ctl->rebuild) return;
  if (blockIdx.x == 0 && threadIdx.x == 0) stamp(g, 4, now_ns());
  const uint32_t n_active = g.ctl->n_active;
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_active; k += gridDim.x * blockDim.x) {
    // the entry and the head of its list together: k is all their addresses need
    const uint2 e = ld_keep(g.nl_active + k);
    int32_t     first4[4];
#pragma unroll
    for (int u = 0; u < 4; u++) first4[u] = ld_keep(g.act_items + int64_t(u) * g.nl_ld + k);
    check_one(s, g, crash_mode, rebounce, k, int64_t(e.x), e.y, first4);
  }
}

// First kernel of every pass, one warp.
//  (1) Sharded runs with peer access: the hand-shake of the pull exchange.  Lane r tells rank r "the positions, group boxes and
//      geometry of my pass number E are in place" (my displacement word first, then — after a system-wide fence — E itself into
//      my slot of r's flag block) and then waits (bounded) until rank r has said the same.  After that every kernel of this pass
//      may read the peers' buffers of the current parity; a peer cannot overwrite them before it has seen THIS rank's pass E + 1.
//      The words travel double-buffered by pass parity; a lost peer counts as "unbounded displacement" and is reported through the
//      mapped status word instead of hanging the GPU.
//  (2) Are the neighbour lists still good for the positions of this pass?  The swarm-wide displacement bound is the largest of
//      every rank's; everything else is as on a single GPU.
__global__ void __launch_bounds__(32) decide_kernel(NlCtl* __restrict__ c, unsigned long long* __restrict__ pair_counter, double skin, int always,
                                                    cudaGraphConditionalHandle handle, int has_handle, P2PCtl p, unsigned long long* tl) {
  const uint32_t full = 0xffffffffu;
  const int      lane = threadIdx.x;
  unsigned long long* row = tl ? tl + (c->n_passes % MRSB_TL_TICKS) * 8 : nullptr;
  if (row && lane == 0) row[0] = now_ns();
  // every load first (they are independent: one round trip), then the decision, then the stores
  uint32_t                 bits  = c->disp_max_bits;  // largest squared displacement of the stepping launch since the last pass (float, rounded up)
  const double             D_old = c->D_total;
  const uint32_t           valid = c->valid;
  const unsigned long long n_rebuilds = c->n_rebuilds, n_passes = c->n_passes;
  if (p.n_ranks > 1) {
    const unsigned long long epoch = c->epoch + 1ull;
    const int                slot  = int(epoch & 1ull);
    const bool               peer  = lane < p.n_ranks && lane != p.rank;
    volatile unsigned long long* theirs = peer ? p.peer_flags[lane] : nullptr;
    if (peer) theirs[p.n_ranks + 2 * p.rank + slot] = (unsigned long long)(always ? 0xFFFFFFFFu : bits);  // a rank without lists cannot bound its displacement
    __threadfence_system();
    if (peer) theirs[p.rank] = epoch;
    if (row && lane == 0) row[1] = now_ns();
    uint32_t got = 0u;
    if (peer) {
      volatile const unsigned long long* mine = p.flags;
      const long long                    t0   = clock64();
      bool                               ok   = true;
      while (mine[lane] < epoch) {
        if (clock64() - t0 > p.budget) {  // a peer is gone; report instead of hanging the GPU
          *p.status = 1;
          ok        = false;
          break;
        }
        __nanosleep(32);
      }
      __threadfence_system();
      got = ok ? uint32_t(mine[p.n_ranks + 2 * lane + slot]) : 0xFFFFFFFFu;
    }
    bits = max(bits, __reduce_max_sync(full, got));
    if (lane == 0) c->epoch = epoch;
  }
  if (lane != 0) return;
  if (row) row[2] = now_ns();
  const double d       = __dsqrt_ru(double(__uint_as_float(bits)));  // NaN stays NaN: an unbounded word rebuilds
  double       D       = __dadd_ru(D_old, d);
  const bool   rebuild = always || !valid || !(__dmul_ru(2.0, D) <= skin);
  if (has_handle) cudaGraphSetConditional(handle, rebuild ? 1u : 0u);
  *pair_counter    = 0ull;  // pairs found by this pass
  c->disp_max_bits = 0u;
  if (rebuild) {
    D            = 0.0;
    c->valid     = 1u;
    c->n_crowded = 0u;  // build_lists_kernel counts them again
    c->n_active  = 0u;  // ... and compact_kernel the UAVs with work
    c->n_rebuilds = n_rebuilds + 1ull;
  }
  if (row) row[5] = rebuild ? 1ull : 0ull;
  c->D_total  = D;
  c->rebuild  = rebuild ? 1u : 0u;
  c->n_passes = n_passes + 1ull;
}

// ---- neighbour observations (mrsb_pack_neighbours_device) -----------------------------------------------
// The k nearest UAVs within a caller-chosen radius, for every UAV of a single-shard handle.  The table is the collision pass'
// (count_kernel, scan_kernel<false>, scatter_kernel) over a workspace of its own — `t` is a DevGrid that holds only the table
// fields — so nothing the collision pass keeps is read or written.  Positions and velocities come from the state rows, not from
// the packed positions, which may be stale or switched off.

// One thread per slot, in tile order (the state loads coalesce); padding slots are skipped.  Writes the positions and velocities in
// external order: the table is built on the former, the query reads the winners' rows from both.
__global__ void __launch_bounds__(256) nb_pack_kernel(DevState s, double* __restrict__ pos, double* __restrict__ vel) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= s.ld) return;
  const int64_t e = s.inv ? int64_t(s.inv[i]) : (i < s.n ? i : -1);
  if (e < 0) return;
#pragma unroll
  for (int c = 0; c < 3; c++) {
    pos[3 * e + c] = s.st[tix(ST_ROWS, c, i)];
    vel[3 * e + c] = s.st[tix(ST_ROWS, 3 + c, i)];
  }
}

// (d2, j) ordering of the neighbour set: ties go to the lower index
DEV bool nb_before(double da, int32_t ja, double db, int32_t jb) { return da < db || (da == db && ja < jb); }

// One thread per record, as collide_kernel (neighbouring threads walk the same cells), for UAV i of the record: every candidate of
// its stencil (the collision pass' layout: 2 x 2 rows of 2 cells of edge 2 * reach) gets the exact predicate d2 < r2 (nf_dist2 with
// dx = x_j - x_i), j != i, and the row check that rejects bucket aliases; the K best by (d2, j) stay in registers (K >= k, sorted,
// unrolled insert).  Positions and velocities of the k winners are fetched after the walk, so a candidate costs one record.
template <int K>
__global__ void __launch_bounds__(128) nb_query_kernel(DevGrid t, int64_t n, const double* __restrict__ pos, const double* __restrict__ vel, double r2,
                                                        int k, int32_t* __restrict__ idx_out, double* __restrict__ rows_out, int64_t stride,
                                                        int32_t* __restrict__ count_out) {
  const int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const double4 q = t.rec[p];  // every UAV is inserted: records [0, n) are the primary ones
  const int64_t i = __double_as_longlong(q.w);
  double        bd[K];
  int32_t       bj[K];
#pragma unroll
  for (int u = 0; u < K; u++) bd[u] = __longlong_as_double(0x7FF0000000000000ll), bj[u] = INT32_MAX;
  int32_t cnt = 0;
  // a UAV with a non-finite position has no neighbours (and is nobody's: its d2 is never < r2)
  if (isfinite(q.x) && isfinite(q.y) && isfinite(q.z)) {
    const Stencil st = stencil_of(t, q.x, q.y, q.z);
    for (int a = 0; a < 4; a++) {
      for (uint32_t r = st.lo[a]; r < st.hi[a]; r++) {
        const double4 c  = t.rec[r];
        const double  d2 = nf_dist2(c.x, c.y, c.z, q.x, q.y, q.z);
        if (!(d2 < r2)) continue;
        const int32_t j = int32_t(__double_as_longlong(c.w));
        if (int64_t(j) == i || cell_of(c.y, t.inv_cell) != st.rcy[a] || cell_of(c.z, t.inv_cell) != st.rcz[a]) continue;  // self, alias
        cnt++;
        if (!nb_before(d2, j, bd[K - 1], bj[K - 1])) continue;
        bd[K - 1] = d2, bj[K - 1] = j;
#pragma unroll
        for (int u = K - 1; u > 0; u--) {
          if (nb_before(bd[u], bj[u], bd[u - 1], bj[u - 1])) {
            const double  td = bd[u];
            const int32_t tj = bj[u];
            bd[u] = bd[u - 1], bj[u] = bj[u - 1];
            bd[u - 1] = td, bj[u - 1] = tj;
          }
        }
      }
    }
  }
  const int m = min(cnt, k);
  if (count_out) count_out[i] = cnt;
  if (idx_out) {
#pragma unroll
    for (int u = 0; u < K; u++)
      if (u < k) idx_out[i * k + u] = u < m ? bj[u] : -1;
  }
  if (rows_out) {
    double*      o  = rows_out + i * stride;
    const double vx = m > 0 ? vel[3 * i] : 0.0, vy = m > 0 ? vel[3 * i + 1] : 0.0, vz = m > 0 ? vel[3 * i + 2] : 0.0;
#pragma unroll
    for (int u = 0; u < K; u++) {
      if (u >= k) break;
      double b[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      if (u < m) {
        const int64_t j = bj[u];
        b[0] = __dsub_rn(pos[3 * j], q.x), b[1] = __dsub_rn(pos[3 * j + 1], q.y), b[2] = __dsub_rn(pos[3 * j + 2], q.z);
        b[3] = __dsub_rn(vel[3 * j], vx), b[4] = __dsub_rn(vel[3 * j + 1], vy), b[5] = __dsub_rn(vel[3 * j + 2], vz);
      }
#pragma unroll
      for (int c = 0; c < 6; c++) o[6 * u + c] = b[c];
    }
  }
}

}  // namespace

int scan_tiles_for(int64_t n_items) {
  return int((n_items + SCAN_TILE - 1) / SCAN_TILE);
}

// table build: [box,] count [, halo count], scan, scatter [, halo scatter].  Returns the number of own kernels.
static int launch_table(const DevState& s, const DevGrid& g, const PeerView& pv, cudaStream_t stream) {
  const int      T      = 256;
  const bool     pull   = pv.n_ranks > 1;
  const int      filter = !pull && s.n_global > s.n;
  const int64_t  j0     = pull ? s.shard_begin : 0;
  const int64_t  cnt    = pull ? s.n : s.n_global;
  const unsigned nb     = unsigned((cnt + T - 1) / T);
  const int64_t  n_scan = int64_t(g.n_buckets) + 3;
  int            own    = 0;
  cudaMemsetAsync(g.count, 0, sizeof(uint32_t) * size_t(n_scan), stream);
  cudaMemsetAsync(g.scan_state, 0, sizeof(unsigned long long) * size_t(2 + g.scan_tiles + scan_tiles_for(s.n)), stream);  // both scans of a rebuild
  if (filter) {
    box_reset_kernel<<<1, 32, 0, stream>>>(g.aabb);
    if (s.n > 0) box_kernel<<<unsigned(std::min<int64_t>((s.n + T - 1) / T, 296)), T, 0, stream>>>(s.gpos, s.shard_begin, s.n, g.aabb);
    own += 2;
  }
  if (pull) {
    cudaMemsetAsync(g.halo_n, 0, 2 * sizeof(uint32_t), stream);  // halo_n and the work-list counter behind it
    box_reset_kernel<<<1, 32, 0, stream>>>(g.aabb);
    const int64_t n_groups = (s.n + 31) / 32;
    if (n_groups > 0) box_from_groups_kernel<<<unsigned(std::min<int64_t>((n_groups + 255) / 256, 148)), 256, 0, stream>>>(s.gbox, n_groups, g.aabb);
    own += 2;
  }
  if (cnt > 0) {
    count_kernel<<<nb, T, 0, stream>>>(s.gpos, j0, cnt, s.shard_begin, s.n, filter, g.aabb, g.n_buckets - 1, g.inv_cell, g.reach, g.count, g.bucket, g.rank);
    own += 1;
  }
  if (pull) {
    int64_t chunks = 0;
    for (int r = 0; r < pv.n_ranks; r++)
      if (r != pv.rank) chunks += ((pv.begin[r + 1] - pv.begin[r] + 31) / 32 + 15) / 16;
    if (chunks > 0) {
      halo_groups_kernel<<<unsigned(std::min<int64_t>((chunks + 7) / 8, 148 * 4)), T, 0, stream>>>(g, pv);
      halo_fetch_kernel<<<148 * 2, T, 0, stream>>>(s, g, pv, g.n_buckets - 1);  // one warp per listed group, grid-stride over the list
      own += 2;
    }
  }
  scan_kernel<false><<<unsigned(g.scan_tiles), 256, 0, stream>>>(g.count, g.begin, n_scan, g.scan_state);
  own += 1;
  if (cnt > 0) {
    scatter_kernel<<<nb, T, 0, stream>>>(s.gpos, j0, cnt, g.bucket, g.rank, g.begin, g.n_buckets, g.rec);
    own += 1;
  }
  if (pull) {
    scatter_halo_kernel<<<unsigned(std::min<int64_t>((g.halo_cap + T - 1) / T, 148 * 4)), T, 0, stream>>>(g);
    own += 1;
  }
  return own;
}

// The full pass of every tick (handles without neighbour lists): [hand-shake,] table + collide_kernel.
int launch_collide(const DevState& s, const DevGrid& g, const PeerView& pv, const P2PCtl& p2p, int crash_mode, double rebounce, cudaStream_t stream) {
  const int64_t n = s.n_global;
  if (n <= 0) return 0;
  int own = 0;
  if (p2p.n_ranks > 1) {
    own += launch_collide_decide(g, p2p, 1, cudaGraphConditionalHandle{}, 0, stream);  // hand-shake; also resets the pair counter
  } else {
    cudaMemsetAsync(g.counters, 0, sizeof(unsigned long long), stream);
  }
  own += launch_table(s, g, pv, stream);
  const int64_t n_rec_max = pv.n_ranks > 1 ? s.n + g.halo_cap : n;
  collide_kernel<<<unsigned((n_rec_max + 127) / 128), 128, 0, stream>>>(s, g, crash_mode, rebounce);
  return own + 1;
}

// ---- the pass with neighbour lists, in three pieces so that api.cu can put the middle one into the
// body of a conditional graph node -----------------------------------------------------------------
int launch_collide_decide(const DevGrid& g, const P2PCtl& p2p, int always, cudaGraphConditionalHandle handle, int has_handle, cudaStream_t stream) {
  decide_kernel<<<1, 32, 0, stream>>>(g.ctl, g.counters, g.skin, always, handle, has_handle, p2p, g.tl);
  return 1;
}
int launch_collide_rebuild(const DevState& s, const DevGrid& g, const PeerView& pv, cudaStream_t stream) {
  if (s.n_global <= 0) return 0;
  const int     own       = launch_table(s, g, pv, stream);
  const int64_t n_rec_max = pv.n_ranks > 1 ? s.n + g.halo_cap : s.n_global;
  build_lists_kernel<<<unsigned(std::max<int64_t>(1, std::min<int64_t>((n_rec_max + 31) / 32, 148 * 16))), 128, 0, stream>>>(s, g);
  if (s.n <= 0) return own + 1;
  // g.rank is free again after the scatter: it takes the slots
  scan_kernel<true><<<unsigned(scan_tiles_for(s.n)), 256, 0, stream>>>(g.nl_count, g.rank, s.n, g.scan_state + 1 + g.scan_tiles);
  compact_kernel<<<unsigned((s.n + 255) / 256), 256, 0, stream>>>(g, g.rank, s.n);
  return own + 3;
}
// list check.  beside_rebuild: captured next to the conditional node (see check_kernel); it then also refreshes the halo first.
int launch_collide_check(const DevState& s, const DevGrid& g, const PeerView& pv, int crash_mode, double rebounce, int beside_rebuild, cudaStream_t stream) {
  if (s.n <= 0) return 0;
  int own = 0;
  if (pv.n_ranks > 1 && beside_rebuild) {
    // between rebuilds: the halo's current positions from their owners (a rebuild fetches them itself)
    refresh_halo_kernel<<<unsigned(std::max<int64_t>(1, std::min<int64_t>((g.halo_cap + 63) / 64, 148 * 2))), 64, 0, stream>>>(s, g, pv);
    own += 1;
  }
  check_kernel<<<unsigned(std::min<int64_t>((s.n + MRSB_CHECK_THREADS - 1) / MRSB_CHECK_THREADS, 148 * MRSB_CHECK_MINB)), MRSB_CHECK_THREADS, 0, stream>>>(s, g, crash_mode, rebounce,
                                                                                                                                                       beside_rebuild);
  return own + 1;
}

// Neighbour observations: pack, table (count, scan, scatter), query.  `t` holds the workspace's table fields; pos / vel the
// workspace's packed rows.  Enqueued on `stream`, no host synchronisation.
int launch_neighbours(const DevState& s, const DevGrid& t, double* pos, double* vel, double r2, int k, int32_t* idx, double* rows, int stride,
                      int32_t* count, cudaStream_t stream) {
  const int64_t n = s.n;
  if (n <= 0) return 0;
  const int      T      = 256;
  const unsigned nb     = unsigned((n + T - 1) / T);
  const int64_t  n_scan = int64_t(t.n_buckets) + 3;
  cudaMemsetAsync(t.count, 0, sizeof(uint32_t) * size_t(n_scan), stream);
  cudaMemsetAsync(t.scan_state, 0, sizeof(unsigned long long) * size_t(1 + t.scan_tiles), stream);
  nb_pack_kernel<<<unsigned((s.ld + T - 1) / T), T, 0, stream>>>(s, pos, vel);
  count_kernel<<<nb, T, 0, stream>>>(pos, 0, n, 0, n, 0, nullptr, t.n_buckets - 1, t.inv_cell, t.reach, t.count, t.bucket, t.rank);
  scan_kernel<false><<<unsigned(t.scan_tiles), 256, 0, stream>>>(t.count, t.begin, n_scan, t.scan_state);
  scatter_kernel<<<nb, T, 0, stream>>>(pos, 0, n, t.bucket, t.rank, t.begin, t.n_buckets, t.rec);
  const unsigned nq = unsigned((n + 127) / 128);
  if (k <= 4) nb_query_kernel<4><<<nq, 128, 0, stream>>>(t, n, pos, vel, r2, k, idx, rows, stride, count);
  else if (k <= 8) nb_query_kernel<8><<<nq, 128, 0, stream>>>(t, n, pos, vel, r2, k, idx, rows, stride, count);
  else nb_query_kernel<MRSB_MAX_NEIGHBOURS><<<nq, 128, 0, stream>>>(t, n, pos, vel, r2, k, idx, rows, stride, count);
  return 5;
}
