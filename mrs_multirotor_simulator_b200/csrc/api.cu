// api.cu — the C ABI of include/mrsb.h: host bookkeeping around the kernels.
// Every entry point cites the reference member it replaces in include/mrsb.h.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "internal.h"
#include "params.h"

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                                              \
  do {                                                                                                        \
    cudaError_t e_ = (call);                                                                                  \
    if (e_ != cudaSuccess) return fail(MRSB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// ------------------------------------------------------------------------------------------
// NCCL, loaded lazily so single-GPU users need no libnccl
// ------------------------------------------------------------------------------------------
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*)                                                         = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int)                                  = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t)                                                            = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t)    = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)()                                                                       = nullptr;
  ncclResult_t (*GroupEnd)()                                                                         = nullptr;
  const char* (*GetErrorString)(ncclResult_t)                                                        = nullptr;
};
static NcclApi g_nccl;

static int load_nccl() {
  if (g_nccl.lib) return MRSB_OK;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void*       lib     = nullptr;
  for (const char* n : names) {
    lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (lib) break;
  }
  if (!lib) return fail(MRSB_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
#define SYM(field, name)                                                          \
  *(void**)(&g_nccl.field) = dlsym(lib, name);                                    \
  if (!g_nccl.field) return fail(MRSB_ERR_NCCL, "libnccl lacks symbol %s", name);
  SYM(GetUniqueId, "ncclGetUniqueId");
  SYM(CommInitRank, "ncclCommInitRank");
  SYM(CommDestroy, "ncclCommDestroy");
  SYM(AllGather, "ncclAllGather");
  SYM(Broadcast, "ncclBroadcast");
  SYM(GroupStart, "ncclGroupStart");
  SYM(GroupEnd, "ncclGroupEnd");
  SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
  g_nccl.lib = lib;
  return MRSB_OK;
}

#define NC(call)                                                                                                  \
  do {                                                                                                            \
    ncclResult_t r_ = (call);                                                                                     \
    if (r_ != ncclSuccess) return fail(MRSB_ERR_NCCL, "%s failed: %s", #call, g_nccl.GetErrorString(r_));          \
  } while (0)

// ------------------------------------------------------------------------------------------
// memory: the one owner of every allocation
// ------------------------------------------------------------------------------------------
// A block of cap() elements of device memory, or of pinned host memory mapped into the device's address space when Pinned.
// Move-only; the destructor frees it.
template <class T, bool Pinned = false>
class Mem {
 public:
  Mem() = default;
  Mem(Mem&& o) noexcept { *this = std::move(o); }
  Mem& operator=(Mem&& o) noexcept {
    release();
    p_ = std::exchange(o.p_, nullptr), cap_ = std::exchange(o.cap_, 0);
    return *this;
  }
  ~Mem() { release(); }

  T*     get() const { return p_; }
  size_t cap() const { return cap_; }

  int alloc(size_t count) {  // in place of the block held so far
    Mem m;
    if (Pinned) {
      CU(cudaHostAlloc(&m.p_, sizeof(T) * count, cudaHostAllocMapped));
    } else {
      CU(cudaMalloc(&m.p_, sizeof(T) * count));
    }
    m.cap_ = count;
    *this  = std::move(m);
    return MRSB_OK;
  }
  // At least `need` elements: a smaller block is replaced by one of `count` >= need elements.  The new block is allocated first;
  // only then is `stream`, where the old block may still be in use, waited for and the old block freed.  A grow that fails
  // leaves the old block and its capacity.
  int grow(size_t need, size_t count, cudaStream_t stream) {
    if (need <= cap_) return MRSB_OK;
    Mem m;
    int rc = m.alloc(count);
    if (rc) return rc;
    if (p_) CU(cudaStreamSynchronize(stream));
    *this = std::move(m);
    return MRSB_OK;
  }

 private:
  void release() {
    if (p_) Pinned ? cudaFreeHost(p_) : cudaFree(p_);
  }
  T*     p_   = nullptr;
  size_t cap_ = 0;
};

// ------------------------------------------------------------------------------------------
// the handle
// ------------------------------------------------------------------------------------------
struct ParamSet {
  mrsb_model_params      mp;
  mrsb_controller_params cp;
};

// Buckets of the tiled arrays: one per airframe type present at create (a single one for a uniform batch), each a whole number
// of tiles, so that the stepping kernel specialised for (motor count, parameter set) runs on each.
#define MAX_BUCKETS 8
struct Bucket {
  int64_t   slot0 = 0, count = 0;  // first slot (multiple of 128), UAVs
  int       nm    = 0;             // n_motors shared by its UAVs, or 0 if mixed (after per-UAV setParams)
  int       pset  = -1;            // parameter set shared by its UAVs, or -1 if mixed
  DevParams params{};              // host copy of that set (goes to the staged kernel by value)
};

// Everything the launches of a collision pass, and of a tick of mrsb_run (stepping launch + pass), take by value.  Those launches
// take their arguments from this value alone, so a captured graph whose key equals what graph_args() gives now replays exactly
// what would be launched now.  graph_args() zeroes it and copies whole structs in: equal keys are equal byte for byte (memcmp).
static_assert(std::is_trivially_copyable_v<DevState> && std::is_trivially_copyable_v<DevGrid> && std::is_trivially_copyable_v<PeerView> &&
              std::is_trivially_copyable_v<P2PCtl> && std::is_trivially_copyable_v<DevParams> && std::is_trivially_copyable_v<Bucket>);
struct GraphArgs {
  DevState s;  // its position buffers are the ones of the pass' parity
  DevGrid  grid;
  PeerView pv;
  P2PCtl   p2p;
  int32_t  crash, lists;
  double   rebounce;
  // the stepping launch (zero in a pass graph's key); publish: publish_positions follows (bucketed pull-exchange handles)
  int32_t with_step, k_substeps, uniform_mode, any_moment, publish, n_buckets;
  double  dt;
  Bucket  buckets[MAX_BUCKETS];
};
static_assert(std::is_trivially_copyable_v<GraphArgs>);

// A captured graph (exec, nullptr if not captured) and the GraphArgs it launches.  Move-only; the destructor destroys the graph.
struct Graph {
  cudaGraphExec_t exec = nullptr;
  int             own  = 0;  // own kernels per replay (for the launch counter)
  GraphArgs       key{};

  Graph() = default;
  explicit Graph(const GraphArgs& a) { std::memcpy(&key, &a, sizeof(a)); }
  Graph(Graph&& o) noexcept { *this = std::move(o); }
  Graph& operator=(Graph&& o) noexcept {
    if (exec) cudaGraphExecDestroy(exec);
    exec = std::exchange(o.exec, nullptr), own = o.own;
    std::memcpy(&key, &o.key, sizeof(key));
    return *this;
  }
  ~Graph() {
    if (exec) cudaGraphExecDestroy(exec);
  }
  bool holds(const GraphArgs& a) const { return std::memcmp(&key, &a, sizeof(a)) == 0; }
};

struct mrsb_sim {
  int          device = 0;
  cudaStream_t stream = nullptr;
  DevState     ds{};
  DevGrid      grid{};
  Mem<int32_t> pairs;  // grid.pairs (mrsb_set_pair_capacity)

  std::vector<ParamSet>      sets;
  std::map<std::string, int> set_index;
  // everything allocated once, at create or by setup_p2p (dalloc), freed by the destructor
  std::vector<Mem<unsigned char>> mem;

  std::vector<int32_t>       pset_host;  // [n_global]
  Mem<DevParams>             d_params;
  Mem<uint8_t>               d_takeoff0;  // initial take-off flag of every set (what a respawn restores)
  int32_t*                   d_pset       = nullptr;
  bool                       params_dirty = true;

  Mem<char>    d_stage;  // staging for payload transposes
  Mem<int32_t> d_idx;

  int  uniform_mode = MRSB_INPUT_UNKNOWN;  // INPUT_MODE shared by all UAVs, or -1 if mixed
  bool any_moment   = false;
  std::vector<Bucket>  buckets;
  std::vector<int32_t> perm_host, inv_host;  // external local index -> slot, slot -> external (-1 = padding); empty = identity
  int32_t*             d_perm = nullptr;
  int32_t*             d_inv  = nullptr;

  int    coll_enabled = 0, coll_crash = 0;
  double coll_rebounce = 0.0;

  double   filt_dt  = -1.0;   // dt the DevParams::filt column of the device table was last prepared for (< 0: stale)
  uint32_t outputs  = MRSB_OUT_IMU | MRSB_OUT_POSITIONS;  // mrsb_set_outputs
  bool     iterate_without_input = true;                  // mrsb_set_iterate_without_input (ROSW:265)
  double*  d_geom[2] = {nullptr, nullptr};                // collision geometry [n_global][4]; [1] only with the pull exchange

  ncclComm_t           comm    = nullptr;
  int                  n_ranks = 1, rank = 0;
  std::vector<int64_t> shard_begin_of, shard_count_of;
  bool                 equal_shards = true;

  // Pull exchange over peer memory (set up by mrsb_comm_init_nccl when every peer is reachable).  Positions, per-group boxes
  // and collision geometry exist twice; collision pass number k (1, 2, ...) READS buffer k & 1 on every rank, and everything
  // that writes positions between pass k - 1 and pass k writes buffer k & 1 — a peer that is still inside pass k - 1 reads the
  // other one, and it cannot be further behind than that (the hand-shake of pass k waits for it).
  bool                 p2p       = false;
  double*              gbuf[2]   = {nullptr, nullptr};
  uint32_t*            d_gbox[2] = {nullptr, nullptr};
  int64_t              pass_no   = 0;      // collision passes done so far (pull exchange)
  bool                 wrote_since_pass = false;  // positions of buffer (pass_no + 1) & 1 are complete
  std::vector<int32_t> pending_geom[2];    // local indices whose geometry changed but is not yet in that buffer (-1 = all)
  PeerView             pv[2]{};            // what the kernels of a pass with parity k read
  PeerView             pv_local{};         // everything in this handle's own arrays
  P2PCtl               p2pctl{};
  unsigned long long*  d_flags   = nullptr;              // this rank's flag block, written by the peers
  unsigned long long** d_peer_flags = nullptr;           // device array [n_ranks] of the peers' flag blocks
  std::vector<void*>   ipc_opened;
  Mem<int, true>       h_status;                         // pinned, mapped: set by the hand-shake on time-out

  // pipelined host I/O (mrsb_set_input_async, mrsb_set_input_rows_async / mrsb_get_positions_async, mrsb_get_observations_async)
  cudaStream_t up_stream = nullptr, down_stream = nullptr;
  Mem<double>  d_up[2];      // staged command rows
  Mem<int32_t> d_up_idx[2];  // beside them, the index list [n] and the mode list [n] of a row upload
  Mem<int32_t> d_last;       // one word per slot: the last row of a row upload addressed to it, -1 between uploads (made on first use)
  Mem<double>  d_snap[2];    // position snapshots [n_local][3]
  Mem<double>  d_obs[2];     // observation snapshots [n_local][17] (made on first use)
  cudaEvent_t  ev_up[2] = {nullptr, nullptr}, ev_applied[2] = {nullptr, nullptr}, ev_snap[2] = {nullptr, nullptr}, ev_down[2] = {nullptr, nullptr};
  cudaEvent_t  ev_obs_snap[2] = {nullptr, nullptr}, ev_obs_down[2] = {nullptr, nullptr};
  uint64_t     n_up = 0, n_down = 0, n_obs = 0;
  Mem<int32_t> d_sub_idx;  // mrsb_set_position_subset: the UAVs the async downloads deliver (its first n_sub; 0: all)
  int64_t      n_sub = 0;

  // the collision pass, and mrsb_run's tick (stepping launch + pass), replayed as CUDA graphs, one per buffer parity (write_buf); with
  // neighbour lists the table rebuild sits in a conditional node.  Captured again when the key is not the GraphArgs of now.
  Graph pass[2], tick[2];
  bool  graph_failed = false;  // a capture failed (e.g. conditional nodes unavailable): no more graphs for this handle

  // neighbour lists (single-shard handles)
  bool     lists_on            = false;
  int      steps_since_pass    = 0;     // stepping launches since the last collision pass
  bool     positions_touched   = true;  // positions were written by something else than ONE stepping launch
  int      rebuild_own         = 0;     // own kernels of one rebuild (for the launch counter)
  int64_t  list_passes         = 0;     // passes that went through decide_kernel (it counts them too: NlCtl::n_passes)
  int64_t  rebuilds_counted    = 0;
  Mem<uint32_t, true> h_one;               // pinned constant 1 (source of the async "force rebuild" copy)
  Mem<unsigned long long, true> h_until;   // pinned source of NlCtl::write_all_until (forces_written)

  // neighbour observations (mrsb_pack_neighbours_device): a table of its own, sized for n_local on the first call
  struct NbWorkspace {
    Mem<double>             pos, vel;  // [n_local][3] packed from the state rows, external order
    Mem<uint32_t>           bucket, rank, count, begin;
    Mem<double4>            rec;
    Mem<unsigned long long> scan;
  } nb;

  // snapshots (mrsb_snapshot_*), by id; ids are not reused
  struct Snapshot {
    Mem<unsigned char> mem;  // rows [SNAP_ROWS][n] doubles | flags uint32 [n] | mode uint8 [n], external order (n = n_local)
    bool    filled       = false;               // saved or uploaded at least once
    int32_t uniform_mode = MRSB_INPUT_UNKNOWN;  // the host hints when it was saved
    bool    any_moment   = false;
  };
  std::map<int32_t, Snapshot> snapshots;
  int32_t                     next_snapshot = 1;

  int64_t n_steps = 0, n_passes = 0, n_launches = 0;
  int     step_info[4] = {0, 0, 0, 0};  // last stepping launch: variant, grid, NM_T, MODE_T (mrsb_get_step_info)
};

static std::string set_key(const ParamSet& s) {
  return std::string(reinterpret_cast<const char*>(&s), sizeof(ParamSet));
}

static int intern_set(mrsb_sim* h, const ParamSet& s) {
  const std::string key = set_key(s);
  auto              it  = h->set_index.find(key);
  if (it != h->set_index.end()) return it->second;
  const int id = int(h->sets.size());
  h->sets.push_back(s);
  h->set_index[key] = id;
  h->params_dirty   = true;
  return id;
}

static int check_params(const mrsb_model_params& p) {
  if (p.n_motors < 1 || p.n_motors > MRSB_MAX_MOTORS) return fail(MRSB_ERR_INVALID, "n_motors=%d outside 1..%d", p.n_motors, MRSB_MAX_MOTORS);
  return MRSB_OK;
}

static ParamSet canonical(const mrsb_model_params& mp, const mrsb_controller_params& cp) {
  ParamSet s;
  std::memset(&s, 0, sizeof(s));  // padding bytes take part in the key
  s.mp.n_motors              = mp.n_motors;
  s.mp.ground_enabled        = mp.ground_enabled != 0;
  s.mp.takeoff_patch_enabled = mp.takeoff_patch_enabled != 0;
  s.mp.g = mp.g, s.mp.mass = mp.mass, s.mp.kf = mp.kf, s.mp.km = mp.km, s.mp.prop_radius = mp.prop_radius, s.mp.arm_length = mp.arm_length;
  s.mp.body_height = mp.body_height, s.mp.motor_time_constant = mp.motor_time_constant, s.mp.max_rpm = mp.max_rpm, s.mp.min_rpm = mp.min_rpm;
  s.mp.air_resistance_coeff = mp.air_resistance_coeff, s.mp.ground_z = mp.ground_z;
  std::memcpy(s.mp.J, mp.J, sizeof(mp.J));
  for (int r = 0; r < 4; r++)
    for (int m = 0; m < mp.n_motors; m++) s.mp.allocation_matrix[r * MRSB_MAX_MOTORS + m] = mp.allocation_matrix[r * MRSB_MAX_MOTORS + m];
  s.cp.mixer_desaturation = cp.mixer_desaturation != 0;
  s.cp.rate_kp = cp.rate_kp, s.cp.rate_kd = cp.rate_kd, s.cp.rate_ki = cp.rate_ki;
  s.cp.att_kp = cp.att_kp, s.cp.att_kd = cp.att_kd, s.cp.att_ki = cp.att_ki, s.cp.att_max_rate_roll_pitch = cp.att_max_rate_roll_pitch,
  s.cp.att_max_rate_yaw = cp.att_max_rate_yaw;
  s.cp.vel_kp = cp.vel_kp, s.cp.vel_kd = cp.vel_kd, s.cp.vel_ki = cp.vel_ki, s.cp.vel_max_acceleration = cp.vel_max_acceleration;
  s.cp.pos_kp = cp.pos_kp, s.cp.pos_kd = cp.pos_kd, s.cp.pos_ki = cp.pos_ki, s.cp.pos_max_velocity = cp.pos_max_velocity;
  return s;
}

// Parameter sets nobody refers to any more (per-UAV edits intern a new set per distinct value): dropped once they are the
// majority, ids renumbered, the whole per-UAV index table uploaded again.
static int collect_param_sets(mrsb_sim* h) {
  const int n_sets = int(h->sets.size());
  if (n_sets <= 32) return MRSB_OK;
  std::vector<int> refs(size_t(n_sets), 0);
  for (int32_t id : h->pset_host) refs[size_t(id)]++;
  int live = 0;
  for (int r : refs) live += r > 0;
  if (2 * live > n_sets) return MRSB_OK;
  std::vector<int>      remap(size_t(n_sets), -1);
  std::vector<ParamSet> kept;
  kept.reserve(size_t(live));
  h->set_index.clear();
  for (int k = 0; k < n_sets; k++) {
    if (!refs[size_t(k)]) continue;
    remap[size_t(k)] = int(kept.size());
    h->set_index[set_key(h->sets[size_t(k)])] = int(kept.size());
    kept.push_back(h->sets[size_t(k)]);
  }
  h->sets.swap(kept);
  for (int32_t& id : h->pset_host) id = remap[size_t(id)];
  CU(cudaMemcpyAsync(h->d_pset, h->pset_host.data(), sizeof(int32_t) * h->pset_host.size(), cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return MRSB_OK;
}

// upload the parameter table if it changed; recompute the launch specialisation hints
static int flush_params(mrsb_sim* h) {
  if (!h->params_dirty) return MRSB_OK;
  int rc = collect_param_sets(h);
  if (rc) return rc;
  const int    n_sets = int(h->sets.size());
  const size_t cap    = size_t(std::max(16, 2 * n_sets));
  rc                  = h->d_params.grow(size_t(n_sets), cap, h->stream);
  if (rc) return rc;
  h->ds.params = h->d_params.get();
  rc           = h->d_takeoff0.grow(size_t(n_sets), cap, h->stream);
  if (rc) return rc;
  std::vector<DevParams> host(n_sets);
  std::vector<uint8_t>   takeoff0(size_t(n_sets), 0);
  for (int k = 0; k < n_sets; k++) {
    mrsb_derive(h->sets[k].mp, h->sets[k].cp, &host[k]);
    takeoff0[size_t(k)] = h->sets[k].mp.takeoff_patch_enabled != 0;
  }
  CU(cudaMemcpyAsync(h->d_params.get(), host.data(), sizeof(DevParams) * n_sets, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->d_takeoff0.get(), takeoff0.data(), size_t(n_sets), cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));  // `host` and `takeoff0` go out of scope
  h->filt_dt = -1.0;                     // DevParams::filt has to be prepared again (ensure_filt)
  for (Bucket& b : h->buckets) {
    int nm = -1, ps = -2;
    for (int64_t k = 0; k < b.count; k++) {
      const int64_t e  = h->inv_host.empty() ? b.slot0 + k : h->inv_host[size_t(b.slot0 + k)];
      const int     id = h->pset_host[size_t(h->ds.shard_begin + e)];
      const int     m  = h->sets[size_t(id)].mp.n_motors;
      if (nm == -1) nm = m;
      if (nm != m) nm = 0;
      if (ps == -2) ps = id;
      if (ps != id) ps = -1;
      if (nm == 0 && ps == -1) break;
    }
    b.nm   = nm > 0 ? nm : 0;
    b.pset = ps >= 0 ? ps : -1;
    if (b.pset >= 0) b.params = host[size_t(b.pset)];
  }
  h->params_dirty = false;
  return MRSB_OK;
}

// DevParams::filt = exp(-dt / tau) for every set, evaluated on the device (the same bits whichever kernel variant reads them);
// the staged kernel takes the batch's one set by value, so its host copy gets the device's result.
static int ensure_filt(mrsb_sim* h, double dt) {
  if (h->filt_dt == dt) return MRSB_OK;
  h->n_launches += launch_prep_params(h->d_params.get(), int(h->sets.size()), dt, h->stream);
  for (Bucket& b : h->buckets)
    if (b.pset >= 0) CU(cudaMemcpyAsync(&b.params.filt, &h->d_params.get()[b.pset].filt, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->filt_dt = dt;
  return MRSB_OK;
}

static int ensure_stage(mrsb_sim* h, size_t bytes) {
  return h->d_stage.grow(bytes, std::max<size_t>(bytes, 1 << 16), h->stream);
}

// copy an index list to the device (nullptr stays nullptr = identity) after validating it
static int stage_idx(mrsb_sim* h, int64_t n, const int32_t* idx, const int32_t** out) {
  *out = nullptr;
  if (n < 0 || n > h->ds.n && !idx) return fail(MRSB_ERR_INVALID, "n=%lld outside 0..%lld", (long long)n, (long long)h->ds.n);
  if (!idx || n == 0) return MRSB_OK;
  for (int64_t k = 0; k < n; k++)
    if (idx[k] < 0 || idx[k] >= h->ds.n) return fail(MRSB_ERR_INVALID, "idx[%lld]=%d outside 0..%lld", (long long)k, idx[k], (long long)h->ds.n - 1);
  int rc = h->d_idx.grow(size_t(n), std::max<size_t>(size_t(n), 1024), h->stream);
  if (rc) return rc;
  CU(cudaMemcpyAsync(h->d_idx.get(), idx, sizeof(int32_t) * n, cudaMemcpyHostToDevice, h->stream));
  *out = h->d_idx.get();
  return MRSB_OK;
}

// n rows of `width` doubles in host memory
struct HostRows {
  const double* rows;
  int           width;
};

// the parts back to back into the staging buffer; dev[k]: where part k went
static int stage_rows(mrsb_sim* h, int64_t n, std::initializer_list<HostRows> parts, const double** dev) {
  size_t total = 0;
  for (const HostRows& p : parts) total += size_t(n) * size_t(p.width);
  int rc = ensure_stage(h, sizeof(double) * total);
  if (rc) return rc;
  double* d = reinterpret_cast<double*>(h->d_stage.get());
  for (const HostRows& p : parts) {
    CU(cudaMemcpyAsync(d, p.rows, sizeof(double) * size_t(n) * size_t(p.width), cudaMemcpyHostToDevice, h->stream));
    *dev++ = d;
    d += size_t(n) * size_t(p.width);
  }
  return MRSB_OK;
}

// Host -> device for n addressed UAVs: the index list (validated), then, unless n == 0, the payload parts, none of which may be
// null.  Nothing is launched.
static int upload(mrsb_sim* h, int64_t n, const int32_t* idx, std::initializer_list<HostRows> parts, const int32_t** d_idx, const double** dev) {
  int rc = stage_idx(h, n, idx, d_idx);
  if (rc || n == 0) return rc;
  for (const HostRows& p : parts)
    if (!p.rows) return fail(MRSB_ERR_INVALID, "null payload");
  return stage_rows(h, n, parts, dev);
}

// Device -> host for n addressed UAVs: the index list (validated), then, unless n == 0, `gather(d_idx, staging)` fills `bytes` of
// the staging buffer, which are copied to `out` once they are complete.
template <class Gather>
static int download(mrsb_sim* h, int64_t n, const int32_t* idx, size_t bytes, void* out, Gather gather) {
  const int32_t* d_idx = nullptr;
  int            rc    = stage_idx(h, n, idx, &d_idx);
  if (rc || n == 0) return rc;
  rc = ensure_stage(h, bytes);
  if (rc) return rc;
  h->n_launches += gather(d_idx, static_cast<void*>(h->d_stage.get()));
  CU(cudaMemcpyAsync(out, h->d_stage.get(), bytes, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return MRSB_OK;
}

#define GUARD(h)                                              \
  if (!(h)) return fail(MRSB_ERR_INVALID, "null handle");     \
  CU(cudaSetDevice((h)->device));

static int64_t round_up(int64_t v, int64_t m) {
  return (v + m - 1) / m * m;
}

// *p = a zeroed device array of `count` (at least one) elements that lives as long as the handle
template <class T>
static int dalloc(mrsb_sim* h, T** p, size_t count) {
  const size_t       bytes = sizeof(T) * std::max<size_t>(count, 1);
  Mem<unsigned char> m;
  int                rc = m.alloc(bytes);
  if (rc) return rc;
  CU(cudaMemset(m.get(), 0, bytes));
  *p = reinterpret_cast<T*>(m.get());
  h->mem.push_back(std::move(m));
  return MRSB_OK;
}

static void note_mode(mrsb_sim* h, int mode, int64_t n, bool all) {
  if (all && n == h->ds.n) {
    h->uniform_mode = mode;
  } else if (n > 0 && h->uniform_mode != mode) {
    h->uniform_mode = -1;
  }
}

static int stride_of(int mode) {
  switch (mode) {
    case MRSB_ACTUATOR_CMD:
      return MRSB_MAX_MOTORS;
    case MRSB_ATTITUDE_CMD:
      return 10;
    case MRSB_TILT_HDG_RATE_CMD:
      return 5;
    default:
      return 4;
  }
}

// ---- collision geometry (arm, propeller radius, mass per UAV): what the collision pass reads of the parameters ----------
// which buffer position / geometry writes go to right now
static int write_buf(const mrsb_sim* h) {
  return h->p2p ? int((h->pass_no + 1) & 1) : 0;
}
// geometry of the addressed local UAVs (idx == nullptr: all of them) from the device tables into buffer `b`
static int apply_geom(mrsb_sim* h, int b, int64_t n, const int32_t* d_idx) {
  h->n_launches += launch_set_geom(h->d_geom[b], n, d_idx, h->ds.shard_begin, h->d_pset, h->d_params.get(), h->stream);
  CU(cudaGetLastError());
  return MRSB_OK;
}
// Geometry of local UAVs changed (d_idx: their local indices on the device, nullptr = all).  The buffer being written gets it now;
// with the pull exchange the other buffer may still be read by a peer that is one pass behind, so it gets it when it becomes
// the write buffer (apply_pending_geom, after the next pass).
static int geometry_changed(mrsb_sim* h, int64_t n, const int32_t* idx, const int32_t* d_idx) {
  const int w  = write_buf(h);
  int       rc = apply_geom(h, w, n, d_idx);
  if (rc || !h->p2p) return rc;
  std::vector<int32_t>& pend = h->pending_geom[w ^ 1];
  if (!idx || (pend.size() == 1 && pend[0] < 0)) {
    pend.assign(1, -1);
  } else {
    pend.insert(pend.end(), idx, idx + n);
  }
  return MRSB_OK;
}
static int apply_pending_geom(mrsb_sim* h, int b) {
  std::vector<int32_t>& pend = h->pending_geom[b];
  if (pend.empty()) return MRSB_OK;
  int rc;
  if (pend[0] < 0) {
    rc = apply_geom(h, b, h->ds.n, nullptr);
  } else {
    const int32_t* d_idx = nullptr;
    rc                   = stage_idx(h, int64_t(pend.size()), pend.data(), &d_idx);
    if (!rc) rc = apply_geom(h, b, int64_t(pend.size()), d_idx);
    if (!rc) CU(cudaStreamSynchronize(h->stream));
  }
  pend.clear();
  return rc;
}

// re-point the addressed UAVs to (possibly new) parameter sets produced by `edit(set, k)`; `value_key(k)` tells edits with the
// same outcome apart from others (UAVs with the same old set and the same 64-bit key share the new set)
template <class Edit, class Key>
static int repoint(mrsb_sim* h, int64_t n, const int32_t* idx, Edit edit, Key value_key) {
  const int32_t* d_idx = nullptr;
  int            rc    = stage_idx(h, n, idx, &d_idx);
  if (rc) return rc;
  if (n == 0) return MRSB_OK;
  std::vector<int32_t>                 ids(static_cast<size_t>(n), 0), olds(static_cast<size_t>(n), 0);
  std::map<std::pair<int, uint64_t>, int> memo;
  bool geometry = false;
  for (int64_t k = 0; k < n; k++) {
    const int64_t i   = idx ? idx[k] : k;
    const int     old = h->pset_host[size_t(h->ds.shard_begin + i)];
    olds[size_t(k)]   = old;
    const auto    key = std::make_pair(old, uint64_t(value_key(k)));
    auto          it  = memo.find(key);
    int           id;
    if (it != memo.end()) {
      id = it->second;
    } else {
      ParamSet s = h->sets[old];
      edit(s, k);
      id        = intern_set(h, canonical(s.mp, s.cp));
      memo[key] = id;
      const mrsb_model_params &a = h->sets[size_t(old)].mp, &b = h->sets[size_t(id)].mp;
      if (a.arm_length != b.arm_length || a.prop_radius != b.prop_radius || a.mass != b.mass) geometry = true;
    }
    ids[size_t(k)]                                 = id;
    h->pset_host[size_t(h->ds.shard_begin + i)] = id;
  }
  if (geometry && h->ds.n_global > h->ds.n && !h->p2p) {
    // the collision pass of the OTHER shards evaluates arm + prop and the rebounce weight of these UAVs (SIM:342,350); only the
    // pull exchange lets them read the owner's values
    for (int64_t k = n - 1; k >= 0; k--) h->pset_host[size_t(h->ds.shard_begin + (idx ? idx[k] : k))] = olds[size_t(k)];  // nothing changed
    return fail(MRSB_ERR_STATE, "arm length / propeller radius / mass of a sharded handle can only change while its peers read them from this "
                                "GPU (exchange mode 2, mrsb_comm_init_nccl with peer access)");
  }
  h->params_dirty = true;
  rc              = ensure_stage(h, sizeof(int32_t) * size_t(n));
  if (rc) return rc;
  CU(cudaMemcpyAsync(h->d_stage.get(), ids.data(), sizeof(int32_t) * size_t(n), cudaMemcpyHostToDevice, h->stream));
  h->n_launches += launch_set_pset(h->d_pset, n, d_idx, h->ds.shard_begin, reinterpret_cast<const int32_t*>(h->d_stage.get()), h->stream);
  CU(cudaStreamSynchronize(h->stream));  // `ids` goes out of scope
  if (geometry) {
    rc = flush_params(h);  // the new sets have to be on the device before the geometry is derived from them
    if (rc) return rc;
    rc = stage_idx(h, n, idx, &d_idx);
    if (rc) return rc;
    rc = geometry_changed(h, n, idx, d_idx);
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));
  }
  return MRSB_OK;
}

// Cell geometry of the spatial hash.  Handles that run the full pass every tick use the smallest cell
// whose half covers the search radius sqrt(3) (4 m: fewest candidates).  Handles that keep neighbour
// lists between rebuilds use a larger cell: the list radius is just under cell / 2, so a larger cell
// buys a larger skin, i.e. fewer rebuilds for more candidates per rebuild.
static void set_collision_geometry(mrsb_sim* h, bool lists) {
  DevGrid& g  = h->grid;
  h->lists_on = lists;
  double cell = lists ? 6.0 : 4.0;
  if (const char* e = getenv("MRSB_COLLISION_CELL")) cell = std::max(3.5, atof(e));
  g.inv_cell = 1.0 / cell;
  g.reach    = 0.5 * cell;
  const double r_list = g.reach * (1.0 - 1e-6);
  g.list_r2  = r_list * r_list;
  g.skin     = (r_list - 1.7320508075688775) * (1.0 - 1e-6);
  h->ds.disp_max       = lists ? &g.ctl->disp_max_bits : nullptr;
  h->positions_touched = true;
}

static void make_local_view(mrsb_sim* h) {
  PeerView& v = h->pv_local;
  v           = PeerView{};
  v.n_ranks   = 1;
  v.rank      = 0;
  v.begin[0]  = 0;
  v.begin[1]  = h->ds.n_global;
  v.pos[0]    = h->ds.gpos;
  v.geom[0]   = h->d_geom[0];
}

// Pull exchange set-up: second copies of the position buffer and the geometry table, per-group boxes, this rank's flag block, and
// IPC mappings of every peer's (handles travel through one NCCL all-gather of raw bytes).
static int setup_p2p(mrsb_sim* h) {
  const int    G     = h->n_ranks;
  const size_t ng    = size_t(h->ds.n_global);
  h->gbuf[0]         = h->ds.gpos;
  int rc             = dalloc(h, &h->gbuf[1], 3 * ng);
  if (rc) return rc;
  CU(cudaMemcpy(h->gbuf[1], h->gbuf[0], sizeof(double) * 3 * ng, cudaMemcpyDeviceToDevice));
  rc = dalloc(h, &h->d_geom[1], 4 * ng);
  if (rc) return rc;
  CU(cudaMemcpy(h->d_geom[1], h->d_geom[0], sizeof(double) * 4 * ng, cudaMemcpyDeviceToDevice));
  for (int k = 0; k < 2; k++) {
    rc = dalloc(h, &h->d_gbox[k], 6 * size_t(h->ds.ld / 32 + 1));  // the stepping kernel writes one row per warp of every tile
    if (rc) return rc;
  }
  rc = dalloc(h, &h->d_flags, 3 * size_t(G));  // pass numbers [G] + displacement words [2G]
  if (rc) return rc;
  rc = h->h_status.alloc(1);
  if (rc) return rc;
  *h->h_status.get() = 0;
  struct Handles {
    cudaIpcMemHandle_t buf[2], box[2], geom[2], flags;
  };
  Handles mine;
  for (int k = 0; k < 2; k++) {
    CU(cudaIpcGetMemHandle(&mine.buf[k], h->gbuf[k]));
    CU(cudaIpcGetMemHandle(&mine.box[k], h->d_gbox[k]));
    CU(cudaIpcGetMemHandle(&mine.geom[k], h->d_geom[k]));
  }
  CU(cudaIpcGetMemHandle(&mine.flags, h->d_flags));
  Mem<Handles> d_all;
  rc = d_all.alloc(size_t(G));
  if (rc) return rc;
  CU(cudaMemcpyAsync(d_all.get() + h->rank, &mine, sizeof(Handles), cudaMemcpyHostToDevice, h->stream));
  NC(g_nccl.AllGather(d_all.get() + h->rank, d_all.get(), sizeof(Handles), ncclChar, h->comm, h->stream));
  std::vector<Handles> all;
  all.resize(static_cast<size_t>(G));
  CU(cudaMemcpyAsync(all.data(), d_all.get(), sizeof(Handles) * G, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  std::vector<unsigned long long*> pflags(static_cast<size_t>(G), nullptr);
  for (int k = 0; k < 2; k++) {
    PeerView& v = h->pv[k];
    v           = PeerView{};
    v.n_ranks   = G;
    v.rank      = h->rank;
    for (int r = 0; r < G; r++) v.begin[r] = h->shard_begin_of[size_t(r)];
    v.begin[G] = h->ds.n_global;
  }
  auto open = [&](const cudaIpcMemHandle_t& hd, void** out) -> int {
    CU(cudaIpcOpenMemHandle(out, hd, cudaIpcMemLazyEnablePeerAccess));
    h->ipc_opened.push_back(*out);
    return MRSB_OK;
  };
  for (int r = 0; r < G; r++) {
    if (r == h->rank) {
      for (int k = 0; k < 2; k++) {
        h->pv[k].pos[r]  = h->gbuf[k];
        h->pv[k].box[r]  = h->d_gbox[k];
        h->pv[k].geom[r] = h->d_geom[k];
      }
      pflags[size_t(r)] = h->d_flags;
      continue;
    }
    void* p = nullptr;
    for (int k = 0; k < 2; k++) {
      rc = open(all[size_t(r)].buf[k], &p);
      if (rc) return rc;
      h->pv[k].pos[r] = static_cast<const double*>(p);
      rc              = open(all[size_t(r)].box[k], &p);
      if (rc) return rc;
      h->pv[k].box[r] = static_cast<const uint32_t*>(p);
      rc              = open(all[size_t(r)].geom[k], &p);
      if (rc) return rc;
      h->pv[k].geom[r] = static_cast<const double*>(p);
    }
    rc = open(all[size_t(r)].flags, &p);
    if (rc) return rc;
    pflags[size_t(r)] = static_cast<unsigned long long*>(p);
  }
  rc = dalloc(h, &h->d_peer_flags, size_t(G));
  if (rc) return rc;
  CU(cudaMemcpy(h->d_peer_flags, pflags.data(), sizeof(unsigned long long*) * G, cudaMemcpyHostToDevice));
  // everybody must have opened everybody's memory before the first hand-shake: one more (tiny) collective
  Mem<unsigned long long> d_tmp;
  rc = d_tmp.alloc(size_t(G));
  if (rc) return rc;
  NC(g_nccl.AllGather(d_tmp.get() + h->rank, d_tmp.get(), sizeof(unsigned long long), ncclChar, h->comm, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->p2pctl.peer_flags = h->d_peer_flags;
  h->p2pctl.flags      = h->d_flags;
  h->p2pctl.n_ranks    = G;
  h->p2pctl.rank       = h->rank;
  h->p2pctl.status     = h->h_status.get();
  {
    const char* e    = getenv("MRSB_P2P_TIMEOUT_MS");
    h->p2pctl.budget = (e ? atoll(e) : 20000LL) * 2000000LL;  // default 20 s at ~2 GHz SM clock
  }
  h->p2p     = true;
  h->pass_no = 0;
  // positions, boxes and geometry of the first pass (number 1) live in buffer 1
  h->ds.gpos = h->gbuf[1];
  h->ds.gbox = h->d_gbox[1];
  h->ds.geom = h->d_geom[1];
  h->n_launches += launch_publish_positions(h->ds, h->stream);
  h->wrote_since_pass = true;
  // remote geometry is read from its owner from now on; the hand-shake also carries every rank's displacement bound, so
  // neighbour lists work across shards
  set_collision_geometry(h, h->grid.nl_count != nullptr);
  CU(cudaStreamSynchronize(h->stream));
  return MRSB_OK;
}

extern "C" {

const char* mrsb_last_error(void) {
  return g_err;
}
int mrsb_version(void) {
  return MRSB_VERSION_MAJOR * 1000 + MRSB_VERSION_MINOR;
}

// ------------------------------------------------------------------------------------------
// lifetime
// ------------------------------------------------------------------------------------------
// Nothing is freed while a stream, a graph or a peer's mapping can still reach it.
int mrsb_destroy(mrsb_handle h) {
  if (!h) return MRSB_OK;
  cudaSetDevice(h->device);
  const cudaStream_t streams[3] = {h->stream, h->up_stream, h->down_stream};
  for (cudaStream_t s : streams)
    if (s) cudaStreamSynchronize(s);
  for (int k = 0; k < 2; k++) h->pass[k] = Graph(), h->tick[k] = Graph();  // the graphs before the memory they launch on
  for (void* p : h->ipc_opened) cudaIpcCloseMemHandle(p);
  if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
  for (int k = 0; k < 2; k++)
    for (cudaEvent_t e : {h->ev_up[k], h->ev_applied[k], h->ev_snap[k], h->ev_down[k], h->ev_obs_snap[k], h->ev_obs_down[k]})
      if (e) cudaEventDestroy(e);
  delete h;  // frees the memory
  for (cudaStream_t s : streams)
    if (s) cudaStreamDestroy(s);
  return MRSB_OK;
}

int mrsb_bucket_layout(int64_t n, int32_t n_types, const int32_t* type_of_local_uav, int32_t* slot_of_uav, int64_t* n_slots, int64_t* bucket_first_slot,
                       int64_t* bucket_count) {
  if (n < 0 || n_types < 1 || (n > 0 && !type_of_local_uav) || !n_slots) return fail(MRSB_ERR_INVALID, "bad argument");
  std::vector<int64_t> per_type(size_t(n_types), 0);
  for (int64_t i = 0; i < n; i++) {
    const int t = type_of_local_uav[i];
    if (t < 0 || t >= n_types) return fail(MRSB_ERR_INVALID, "type_of_uav of local UAV %lld is %d, outside 0..%d", (long long)i, t, n_types - 1);
    per_type[size_t(t)]++;
  }
  int present = 0;
  for (int64_t c : per_type) present += c > 0;
  for (int t = 0; t < n_types; t++) {
    if (bucket_first_slot) bucket_first_slot[t] = -1;
    if (bucket_count) bucket_count[t] = per_type[size_t(t)];
  }
  if (present < 2 || present > MAX_BUCKETS || getenv("MRSB_NO_BUCKETS")) {
    // one airframe (or too many to launch one kernel each): slots in the caller's order
    *n_slots = std::max<int64_t>(MRSB_TILE, round_up(n, MRSB_TILE));
    for (int64_t i = 0; i < n && slot_of_uav; i++) slot_of_uav[i] = int32_t(i);
    for (int t = 0; t < n_types && bucket_first_slot; t++)
      if (per_type[size_t(t)] && present == 1) bucket_first_slot[t] = 0;
    return 1;
  }
  std::vector<int64_t> next(size_t(n_types), 0);
  int64_t              slot = 0;
  for (int t = 0; t < n_types; t++) {
    if (!per_type[size_t(t)]) continue;
    next[size_t(t)] = slot;
    if (bucket_first_slot) bucket_first_slot[t] = slot;
    slot += round_up(per_type[size_t(t)], MRSB_TILE);
  }
  *n_slots = slot;
  for (int64_t i = 0; i < n && slot_of_uav; i++) slot_of_uav[i] = int32_t(next[size_t(type_of_local_uav[i])]++);
  return present;
}

int mrsb_create(const mrsb_create_info* info, mrsb_handle* out) {
  if (!info || !out) return fail(MRSB_ERR_INVALID, "null argument");
  *out = nullptr;
  if (info->n_types < 1 || !info->types) return fail(MRSB_ERR_INVALID, "need at least one airframe type");
  if (info->n_local < 0 || info->n_global < info->n_local || info->shard_begin < 0 || info->shard_begin + info->n_local > info->n_global)
    return fail(MRSB_ERR_INVALID, "inconsistent shard: n_local=%lld n_global=%lld shard_begin=%lld", (long long)info->n_local,
                (long long)info->n_global, (long long)info->shard_begin);
  if (info->n_global > 0x7fffffffLL) return fail(MRSB_ERR_INVALID, "n_global exceeds int32 indices");
  for (int t = 0; t < info->n_types; t++) {
    const int rc = check_params(info->types[t]);
    if (rc) return rc;
  }
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) return fail(MRSB_ERR_CUDA, "no CUDA device available (libmrsb has no CPU fallback)");
  if (info->device < 0 || info->device >= n_dev) return fail(MRSB_ERR_INVALID, "device %d outside 0..%d", info->device, n_dev - 1);

  std::unique_ptr<mrsb_sim, int (*)(mrsb_handle)> guard(new mrsb_sim(), mrsb_destroy);  // destroys what a failed create made
  mrsb_sim* h = guard.get();
  h->device   = info->device;
  CU(cudaSetDevice(h->device));
  CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));

  DevState& s   = h->ds;
  s.n           = info->n_local;
  s.n_global    = info->n_global;
  s.shard_begin = info->shard_begin;
  s.n_groups32  = (s.n + 31) / 32;
  // Buckets: the local UAVs sorted (stably) by airframe type, every type padded to whole 128-UAV tiles (mrsb_bucket_layout)
  {
    std::vector<int32_t> type_local(size_t(std::max<int64_t>(s.n, 1)), 0);
    for (int64_t i = 0; i < s.n; i++) type_local[size_t(i)] = info->type_of_uav ? info->type_of_uav[s.shard_begin + i] : 0;
    std::vector<int64_t> first(size_t(info->n_types), -1), count(size_t(info->n_types), 0);
    std::vector<int32_t> slot_of(size_t(std::max<int64_t>(s.n, 1)), 0);
    int64_t              n_slots   = 0;
    const int            n_buckets = mrsb_bucket_layout(s.n, info->n_types, type_local.data(), slot_of.data(), &n_slots, first.data(), count.data());
    if (n_buckets < 0) return n_buckets;
    s.ld = n_slots;
    if (n_buckets > 1) {
      for (int t = 0; t < info->n_types; t++) {
        if (first[size_t(t)] < 0) continue;
        Bucket b;
        b.slot0 = first[size_t(t)], b.count = count[size_t(t)];
        h->buckets.push_back(b);
      }
      h->perm_host.assign(slot_of.begin(), slot_of.begin() + s.n);
      h->inv_host.assign(size_t(s.ld), -1);
      for (int64_t i = 0; i < s.n; i++) h->inv_host[size_t(slot_of[size_t(i)])] = int32_t(i);
    } else {
      Bucket b;
      b.slot0 = 0, b.count = s.n;
      h->buckets.push_back(b);
    }
  }
  const size_t ld = size_t(s.ld);
  int          rc = MRSB_OK;
  if (!h->perm_host.empty()) {
    rc = dalloc(h, &h->d_perm, size_t(s.n));
    if (!rc) rc = dalloc(h, &h->d_inv, ld);
    if (rc) return rc;
    CU(cudaMemcpy(h->d_perm, h->perm_host.data(), sizeof(int32_t) * size_t(s.n), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h->d_inv, h->inv_host.data(), sizeof(int32_t) * ld, cudaMemcpyHostToDevice));
    s.perm = h->d_perm;
    s.inv  = h->d_inv;
  }
  rc = dalloc(h, &s.st, 18 * ld);
  if (!rc) rc = dalloc(h, &s.vprev, 3 * ld);
  if (!rc) rc = dalloc(h, &s.rpm, MRSB_NM * ld);
  if (!rc) rc = dalloc(h, &s.pid, PID_ROWS * ld);
  if (!rc) rc = dalloc(h, &s.fext, 3 * ld);
  if (!rc) rc = dalloc(h, &s.mext, 3 * ld);
  if (!rc) rc = dalloc(h, &s.imu, 3 * ld);
  if (!rc) rc = dalloc(h, &s.initz, ld);
  if (!rc) rc = dalloc(h, &s.cmd, CMD_ROWS * ld);
  if (!rc) rc = dalloc(h, &s.ff, FF_ROWS * ld);
  if (!rc) rc = dalloc(h, &s.flags, ld);
  if (!rc) rc = dalloc(h, &s.mode, ld);
  if (!rc) rc = dalloc(h, &s.gpos, 3 * size_t(s.n_global));
  if (!rc) rc = dalloc(h, &h->d_pset, size_t(s.n_global));
  if (rc) return rc;
  s.pset = h->d_pset;

  // parameter sets: one per airframe type with default controller gains (US:159-169)
  mrsb_controller_params cp;
  mrsb_controller_params_default(&cp);
  std::vector<int> set_of_type(info->n_types);
  for (int t = 0; t < info->n_types; t++) set_of_type[t] = intern_set(h, canonical(info->types[t], cp));
  h->pset_host.resize(size_t(s.n_global));
  for (int64_t j = 0; j < s.n_global; j++) {
    const int t = info->type_of_uav ? info->type_of_uav[j] : 0;
    if (t < 0 || t >= info->n_types) return fail(MRSB_ERR_INVALID, "type_of_uav[%lld]=%d outside 0..%d", (long long)j, t, info->n_types - 1);
    h->pset_host[size_t(j)] = set_of_type[t];
  }
  CU(cudaMemcpy(h->d_pset, h->pset_host.data(), sizeof(int32_t) * size_t(s.n_global), cudaMemcpyHostToDevice));
  rc = flush_params(h);
  if (rc) return rc;
  // collision geometry of the whole swarm (the airframe of every UAV is known everywhere at create time)
  rc = dalloc(h, &h->d_geom[0], 4 * size_t(s.n_global));
  if (rc) return rc;
  s.geom = h->d_geom[0];
  h->n_launches += launch_set_geom(h->d_geom[0], s.n_global, nullptr, 0, h->d_pset, h->d_params.get(), h->stream);
  s.opts = STEP_OPT_IMU | STEP_OPT_GPOS;

  // initial state (MM:183-198 + setStatePos MM:439-446): R = Rz(-heading), flags from the airframe
  {
    std::vector<uint32_t> fl(ld, 0u);
    for (int64_t i = 0; i < s.n; i++)
      fl[h->perm_host.empty() ? size_t(i) : size_t(h->perm_host[size_t(i)])] =
          h->sets[h->pset_host[size_t(s.shard_begin + i)]].mp.takeoff_patch_enabled ? FLAG_TAKEOFF : 0u;
    CU(cudaMemcpy(s.flags, fl.data(), sizeof(uint32_t) * ld, cudaMemcpyHostToDevice));
    const size_t bytes = sizeof(double) * 4 * size_t(std::max<int64_t>(s.n, 1));
    rc                 = ensure_stage(h, bytes);
    if (rc) return rc;
    double* d_xyz = nullptr;
    double* d_hdg = nullptr;
    if (info->spawn_xyz && s.n) {
      d_xyz = reinterpret_cast<double*>(h->d_stage.get());
      CU(cudaMemcpyAsync(d_xyz, info->spawn_xyz, sizeof(double) * 3 * s.n, cudaMemcpyHostToDevice, h->stream));
    }
    if (info->spawn_heading && s.n) {
      d_hdg = reinterpret_cast<double*>(h->d_stage.get()) + 3 * s.n;
      CU(cudaMemcpyAsync(d_hdg, info->spawn_heading, sizeof(double) * s.n, cudaMemcpyHostToDevice, h->stream));
    }
    h->n_launches += launch_set_state_pos(s, s.n, nullptr, d_xyz, d_hdg, h->stream);
    CU(cudaStreamSynchronize(h->stream));
  }

  // collision workspace
  {
    DevGrid&     g  = h->grid;
    const size_t ng = size_t(std::max<int64_t>(s.n_global, 1));
    // >= 1.5 buckets per inserted UAV.  A shard inserts its own UAVs plus the halo of remote ones near its bounding box; the
    // table is sized for a halo of a quarter of the shard (spatially coherent shards have far less; a fuller table only means
    // longer bucket lists, never wrong results).  The table is cleared and prefix-summed at every rebuild, so it should not be
    // larger than it has to be.
    const size_t own    = size_t(std::max<int64_t>(s.n, 1));
    const size_t expect = std::max<size_t>(std::min(ng, own + own / 4 + 4096), 512);
    uint32_t     bits   = 10;
    while (2 * (size_t(1) << bits) < 3 * expect && bits < 30) bits++;
    g.bits      = bits;
    g.n_buckets = 1u << bits;
    g.pair_cap   = int64_t(std::max<size_t>(4096, 4 * size_t(std::max<int64_t>(s.n, 1))));
    g.scan_tiles = scan_tiles_for(int64_t(g.n_buckets) + 3);
    g.halo_cap   = std::max<int64_t>(s.n_global - s.n, 1);  // remote UAVs a rebuild fetches from their owners (pull exchange): at most all of them
    rc = dalloc(h, &g.bucket, ng);
    if (!rc) rc = dalloc(h, &g.rank, ng);
    if (!rc) rc = dalloc(h, &g.count, size_t(g.n_buckets) + 4);  // + mirrors of buckets 0 and 1 + sentinel
    if (!rc) rc = dalloc(h, &g.begin, size_t(g.n_buckets) + 4);
    if (!rc) rc = dalloc(h, &g.aabb, 6);
    if (!rc) rc = dalloc(h, &g.rec, 2 * ng);  // worst case: every UAV in bucket 0 and mirrored
    if (!rc) rc = h->pairs.grow(2 * size_t(g.pair_cap), 2 * size_t(g.pair_cap), h->stream);
    if (!rc) rc = dalloc(h, &g.counters, 4);
    if (!rc) rc = dalloc(h, &g.scan_state, size_t(g.scan_tiles) + size_t(scan_tiles_for(s.n)) + 2);  // table scan + compaction scan
    if (!rc && s.n_global > s.n) rc = dalloc(h, &g.halo_rec, size_t(g.halo_cap));
    if (!rc && s.n_global > s.n) rc = dalloc(h, &g.halo_bucket, size_t(g.halo_cap));
    if (!rc && s.n_global > s.n) rc = dalloc(h, &g.halo_rank, size_t(g.halo_cap));
    if (!rc) rc = dalloc(h, &g.halo_n, 2);
    if (!rc && s.n_global > s.n) rc = dalloc(h, &g.halo_work, size_t(g.halo_cap / 32 + MRSB_MAX_RANKS + 1));
    if (!rc && getenv("MRSB_TIMELINE")) rc = dalloc(h, &g.tl, size_t(MRSB_TL_TICKS) * 8);
    if (!rc) rc = dalloc(h, &g.ctl, 1);
    if (!rc) rc = h->h_one.alloc(2);
    if (!rc) rc = h->h_until.alloc(1);
    if (rc) return rc;
    g.pairs       = h->pairs.get();
    g.halo_work_n = g.halo_n + 1;
    h->h_one.get()[0] = 1u;
    h->h_one.get()[1] = 0xFFFFFFFFu;  // "unbounded displacement"
    // neighbour lists: single-shard handles now, sharded ones once the pull exchange is up (setup_p2p)
    if (s.n > 0 && !getenv("MRSB_NO_NEIGHBOUR_LISTS")) {
      g.nl_ld = s.ld;
      rc      = dalloc(h, &g.nl_count, size_t(g.nl_ld));
      if (!rc) rc = dalloc(h, &g.nl_items, size_t(MRSB_NL_CAP) * size_t(g.nl_ld));
      if (!rc) rc = dalloc(h, &g.nl_active, size_t(g.nl_ld));
      if (!rc) rc = dalloc(h, &g.act_items, size_t(MRSB_NL_CAP) * size_t(g.nl_ld));
      if (rc) return rc;
    }
    set_collision_geometry(h, g.nl_count != nullptr && s.n_global == s.n);
  }
  make_local_view(h);
  h->shard_begin_of = {s.shard_begin};
  h->shard_count_of = {s.n};
  CU(cudaStreamSynchronize(h->stream));
  *out = guard.release();
  return MRSB_OK;
}

int mrsb_sync(mrsb_handle h) {
  GUARD(h);
  CU(cudaStreamSynchronize(h->stream));
  if (h->up_stream) CU(cudaStreamSynchronize(h->up_stream));
  if (h->down_stream) CU(cudaStreamSynchronize(h->down_stream));
  return MRSB_OK;
}

// Streams, events and snapshot buffers of the pipelined host I/O, made on first use.  A call that fails half-way keeps what it
// made and the next one makes the rest: the pipeline is ready once the last of them, d_snap[1], exists.
static int ensure_pipeline(mrsb_sim* h) {
  if (h->d_snap[1].get()) return MRSB_OK;
  for (cudaStream_t* s : {&h->up_stream, &h->down_stream})
    if (!*s) CU(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking));
  const size_t snap = 3 * size_t(std::max<int64_t>(h->ds.n, 1));
  for (int k = 0; k < 2; k++) {
    for (cudaEvent_t* e : {&h->ev_up[k], &h->ev_applied[k], &h->ev_snap[k], &h->ev_down[k]})
      if (!*e) CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    int rc = h->d_snap[k].grow(snap, snap, h->down_stream);
    if (rc) return rc;
  }
  return MRSB_OK;
}

// Room for `rows` doubles and `words` int32 in both staging buffers of the upload ring.  Growing first waits for everything that may
// still use them (the stream applies them, the upload stream fills them), then starts the ring afresh.
static int reserve_upload(mrsb_sim* h, size_t rows, size_t words) {
  if (rows <= std::min(h->d_up[0].cap(), h->d_up[1].cap()) && words <= std::min(h->d_up_idx[0].cap(), h->d_up_idx[1].cap())) return MRSB_OK;
  CU(cudaStreamSynchronize(h->stream));     // the scatter reads the staging buffers,
  CU(cudaStreamSynchronize(h->up_stream));  // the uploads write them
  for (int k = 0; k < 2; k++) {
    int rc = h->d_up[k].grow(rows, rows, h->up_stream);
    if (!rc) rc = h->d_up_idx[k].grow(words, words, h->up_stream);
    if (rc) return rc;
  }
  h->n_up = 0;
  return MRSB_OK;
}

// The snapshot buffers and events of mrsb_get_observations_async on top of ensure_pipeline, made on first use; ready once the last
// of them, d_obs[1], exists.  Sized for every local UAV, so that a position subset never makes them grow.
static int ensure_obs_pipeline(mrsb_sim* h) {
  if (h->d_obs[1].get()) return MRSB_OK;
  int rc = ensure_pipeline(h);
  if (rc) return rc;
  const size_t rows = 17 * size_t(std::max<int64_t>(h->ds.n, 1));
  for (int k = 0; k < 2; k++) {
    for (cudaEvent_t* e : {&h->ev_obs_snap[k], &h->ev_obs_down[k]})
      if (!*e) CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    rc = h->d_obs[k].grow(rows, rows, h->down_stream);
    if (rc) return rc;
  }
  return MRSB_OK;
}

int mrsb_set_input_async(mrsb_handle h, int32_t mode, const double* payload, int32_t stride) {
  GUARD(h);
  if (mode <= MRSB_INPUT_UNKNOWN || mode > MRSB_POSITION_CMD) return fail(MRSB_ERR_INVALID, "mode %d carries no payload", mode);
  if (!payload) return fail(MRSB_ERR_INVALID, "null payload");
  if (stride < (mode == MRSB_ACTUATOR_CMD ? 1 : stride_of(mode))) return fail(MRSB_ERR_INVALID, "stride %d too small for mode %d", stride, mode);
  int rc = ensure_pipeline(h);
  if (rc) return rc;
  const int64_t n     = h->ds.n;
  const size_t  count = size_t(n) * size_t(stride);
  rc                  = reserve_upload(h, count, 0);
  if (rc) return rc;
  const int k = int(h->n_up & 1);
  if (h->n_up >= 2) CU(cudaStreamWaitEvent(h->up_stream, h->ev_applied[k], 0));  // the staging buffer was consumed two uploads ago
  CU(cudaMemcpyAsync(h->d_up[k].get(), payload, sizeof(double) * count, cudaMemcpyHostToDevice, h->up_stream));
  CU(cudaEventRecord(h->ev_up[k], h->up_stream));
  CU(cudaStreamWaitEvent(h->stream, h->ev_up[k], 0));
  h->n_launches += launch_scatter_input(h->ds, mode, n, nullptr, h->d_up[k].get(), stride, h->stream);
  CU(cudaEventRecord(h->ev_applied[k], h->stream));
  h->n_up++;
  note_mode(h, mode, n, true);
  CU(cudaGetLastError());
  return MRSB_OK;
}

// The same ring as mrsb_set_input_async: index list, mode list and rows go into staging buffer n_up & 1, which the stream has
// finished reading two uploads ago; the stream waits for the copies, then the claim and apply kernels resolve duplicate UAVs.
int mrsb_set_input_rows_async(mrsb_handle h, int64_t n, const int32_t* idx, const int32_t* modes, const double* payload, int32_t stride) {
  GUARD(h);
  if (n < 0 || n > INT32_MAX) return fail(MRSB_ERR_INVALID, "n=%lld outside 0..%d", (long long)n, INT32_MAX);
  if (n == 0) return MRSB_OK;
  if (!idx || !modes || !payload) return fail(MRSB_ERR_INVALID, "null idx, modes or payload");
  bool uniform = true;  // every row carries the batch's single mode
  for (int64_t k = 0; k < n; k++) {
    if (idx[k] < 0 || idx[k] >= h->ds.n) return fail(MRSB_ERR_INVALID, "idx[%lld]=%d outside 0..%lld", (long long)k, idx[k], (long long)h->ds.n - 1);
    const int m = modes[k];
    if (m <= MRSB_INPUT_UNKNOWN || m > MRSB_POSITION_CMD) return fail(MRSB_ERR_INVALID, "modes[%lld]=%d carries no payload", (long long)k, m);
    if (stride < (m == MRSB_ACTUATOR_CMD ? 1 : stride_of(m))) return fail(MRSB_ERR_INVALID, "stride %d too small for modes[%lld]=%d", stride, (long long)k, m);
    uniform = uniform && m == h->uniform_mode;
  }
  int rc = ensure_pipeline(h);
  if (rc) return rc;
  if (!h->d_last.get()) {
    const size_t slots = size_t(std::max<int64_t>(h->ds.ld, 1));
    rc                 = h->d_last.alloc(slots);
    if (rc) return rc;
    CU(cudaMemsetAsync(h->d_last.get(), 0xFF, sizeof(int32_t) * slots, h->stream));  // -1 everywhere
  }
  const size_t rows = size_t(n) * size_t(stride);
  rc                = reserve_upload(h, rows, 2 * size_t(n));
  if (rc) return rc;
  const int k = int(h->n_up & 1);
  if (h->n_up >= 2) CU(cudaStreamWaitEvent(h->up_stream, h->ev_applied[k], 0));  // the staging buffer was consumed two uploads ago
  int32_t* d_idx = h->d_up_idx[k].get();
  CU(cudaMemcpyAsync(d_idx, idx, sizeof(int32_t) * size_t(n), cudaMemcpyHostToDevice, h->up_stream));
  CU(cudaMemcpyAsync(d_idx + n, modes, sizeof(int32_t) * size_t(n), cudaMemcpyHostToDevice, h->up_stream));
  CU(cudaMemcpyAsync(h->d_up[k].get(), payload, sizeof(double) * rows, cudaMemcpyHostToDevice, h->up_stream));
  CU(cudaEventRecord(h->ev_up[k], h->up_stream));
  CU(cudaStreamWaitEvent(h->stream, h->ev_up[k], 0));
  h->n_launches += launch_input_rows(h->ds, n, d_idx, d_idx + n, h->d_up[k].get(), stride, h->d_last.get(), h->stream);
  CU(cudaEventRecord(h->ev_applied[k], h->stream));
  h->n_up++;
  if (!uniform) h->uniform_mode = -1;  // rows never make a batch uniform: only a whole-batch call does
  CU(cudaGetLastError());
  return MRSB_OK;
}

int mrsb_get_positions_async(mrsb_handle h, double* out_xyz) {
  GUARD(h);
  if (!out_xyz) return fail(MRSB_ERR_INVALID, "null output");
  int rc = ensure_pipeline(h);
  if (rc) return rc;
  const int    k     = int(h->n_down & 1);
  const size_t bytes = sizeof(double) * 3 * size_t(h->n_sub ? h->n_sub : h->ds.n);
  if (h->n_down >= 2) CU(cudaStreamWaitEvent(h->stream, h->ev_down[k], 0));  // the snapshot buffer was downloaded two reads ago
  if (!(h->ds.opts & STEP_OPT_GPOS)) return fail(MRSB_ERR_STATE, "packed positions are switched off (mrsb_set_outputs)");
  // pull exchange: the buffer being written holds the latest positions only once something wrote it since the last pass
  const double* latest = (h->p2p && !h->wrote_since_pass) ? h->gbuf[h->pass_no & 1] : h->ds.gpos;
  if (h->n_sub) {
    h->n_launches += launch_gather_xyz(latest + 3 * h->ds.shard_begin, h->n_sub, h->d_sub_idx.get(), h->d_snap[k].get(), h->stream);
  } else {
    CU(cudaMemcpyAsync(h->d_snap[k].get(), latest + 3 * h->ds.shard_begin, bytes, cudaMemcpyDeviceToDevice, h->stream));
  }
  CU(cudaEventRecord(h->ev_snap[k], h->stream));
  CU(cudaStreamWaitEvent(h->down_stream, h->ev_snap[k], 0));
  CU(cudaMemcpyAsync(out_xyz, h->d_snap[k].get(), bytes, cudaMemcpyDeviceToHost, h->down_stream));
  CU(cudaEventRecord(h->ev_down[k], h->down_stream));
  h->n_down++;
  return MRSB_OK;
}

// The protocol of mrsb_get_positions_async with a ring of its own: observe_kernel packs the rows into snapshot buffer n_obs & 1, which
// the download stream finished copying out two reads ago, and the download stream copies them out once they are complete.
int mrsb_get_observations_async(mrsb_handle h, double* out17) {
  GUARD(h);
  if (!out17) return fail(MRSB_ERR_INVALID, "null output");
  if (!(h->ds.opts & STEP_OPT_IMU)) return fail(MRSB_ERR_STATE, "the IMU rows are switched off (mrsb_set_outputs)");
  int rc = flush_params(h);  // the range rows read ground_z
  if (!rc) rc = ensure_obs_pipeline(h);
  if (rc) return rc;
  const int     k = int(h->n_obs & 1);
  const int64_t m = h->n_sub ? h->n_sub : h->ds.n;
  if (h->n_obs >= 2) CU(cudaStreamWaitEvent(h->stream, h->ev_obs_down[k], 0));  // the snapshot buffer was downloaded two reads ago
  h->n_launches += launch_observe(h->ds, 3, m, h->n_sub ? h->d_sub_idx.get() : nullptr, h->d_obs[k].get(), 17, h->stream);
  CU(cudaEventRecord(h->ev_obs_snap[k], h->stream));
  CU(cudaStreamWaitEvent(h->down_stream, h->ev_obs_snap[k], 0));
  CU(cudaMemcpyAsync(out17, h->d_obs[k].get(), sizeof(double) * 17 * size_t(m), cudaMemcpyDeviceToHost, h->down_stream));
  CU(cudaEventRecord(h->ev_obs_down[k], h->down_stream));
  h->n_obs++;
  CU(cudaGetLastError());
  return MRSB_OK;
}

int mrsb_set_position_subset(mrsb_handle h, int64_t n, const int32_t* idx) {
  GUARD(h);
  if (h->down_stream) CU(cudaStreamSynchronize(h->down_stream));
  CU(cudaStreamSynchronize(h->stream));
  h->n_sub = 0;
  if (!idx || n <= 0) return MRSB_OK;  // back to "all of them"
  for (int64_t k = 0; k < n; k++)
    if (idx[k] < 0 || idx[k] >= h->ds.n) return fail(MRSB_ERR_INVALID, "idx[%lld]=%d outside 0..%lld", (long long)k, idx[k], (long long)h->ds.n - 1);
  if (n > h->ds.n) return fail(MRSB_ERR_INVALID, "a subset of more than n_local UAVs");
  int rc = h->d_sub_idx.grow(size_t(n), size_t(n), h->stream);
  if (rc) return rc;
  CU(cudaMemcpy(h->d_sub_idx.get(), idx, sizeof(int32_t) * size_t(n), cudaMemcpyHostToDevice));
  h->n_sub = n;
  return MRSB_OK;
}

int mrsb_wait_uploads(mrsb_handle h) {
  GUARD(h);
  if (h->up_stream) CU(cudaStreamSynchronize(h->up_stream));
  return MRSB_OK;
}
int mrsb_wait_downloads(mrsb_handle h) {
  GUARD(h);
  if (h->down_stream) CU(cudaStreamSynchronize(h->down_stream));
  return MRSB_OK;
}
int64_t mrsb_n_local(mrsb_handle h) {
  return h ? h->ds.n : -1;
}
int64_t mrsb_n_global(mrsb_handle h) {
  return h ? h->ds.n_global : -1;
}
void* mrsb_get_stream(mrsb_handle h) {
  return h ? (void*)h->stream : nullptr;
}

// ------------------------------------------------------------------------------------------
// commands
// ------------------------------------------------------------------------------------------
int mrsb_set_input_device(mrsb_handle h, int32_t mode, int64_t n, const int32_t* idx_dev, const double* payload_dev, int32_t stride) {
  GUARD(h);
  if (mode < MRSB_INPUT_UNKNOWN || mode > MRSB_POSITION_CMD) return fail(MRSB_ERR_INVALID, "mode %d is not an INPUT_MODE", mode);
  if (n < 0 || (!idx_dev && n > h->ds.n)) return fail(MRSB_ERR_INVALID, "n=%lld outside 0..%lld", (long long)n, (long long)h->ds.n);
  if (mode == MRSB_INPUT_UNKNOWN) {
    h->n_launches += launch_set_mode(h->ds, n, idx_dev, mode, h->stream);
  } else {
    if (!payload_dev) return fail(MRSB_ERR_INVALID, "null payload");
    if (stride < (mode == MRSB_ACTUATOR_CMD ? 1 : stride_of(mode))) return fail(MRSB_ERR_INVALID, "stride %d too small for mode %d", stride, mode);
    h->n_launches += launch_scatter_input(h->ds, mode, n, idx_dev, payload_dev, stride, h->stream);
  }
  note_mode(h, mode, n, idx_dev == nullptr);
  CU(cudaGetLastError());
  return MRSB_OK;
}

int mrsb_set_input(mrsb_handle h, int32_t mode, int64_t n, const int32_t* idx, const double* payload, int32_t stride) {
  GUARD(h);
  if (mode < MRSB_INPUT_UNKNOWN || mode > MRSB_POSITION_CMD) return fail(MRSB_ERR_INVALID, "mode %d is not an INPUT_MODE", mode);
  const int32_t* d_idx = nullptr;
  int            rc    = stage_idx(h, n, idx, &d_idx);
  if (rc) return rc;
  if (mode == MRSB_INPUT_UNKNOWN) {
    h->n_launches += launch_set_mode(h->ds, n, d_idx, mode, h->stream);
    note_mode(h, mode, n, idx == nullptr);
    return MRSB_OK;
  }
  if (!payload && n) return fail(MRSB_ERR_INVALID, "null payload");
  if (stride < (mode == MRSB_ACTUATOR_CMD ? 1 : stride_of(mode))) return fail(MRSB_ERR_INVALID, "stride %d too small for mode %d", stride, mode);
  if (n == 0) return MRSB_OK;
  const double* d_rows = nullptr;
  rc                   = stage_rows(h, n, {{payload, stride}}, &d_rows);
  if (rc) return rc;
  h->n_launches += launch_scatter_input(h->ds, mode, n, d_idx, d_rows, stride, h->stream);
  note_mode(h, mode, n, idx == nullptr);
  CU(cudaGetLastError());
  return MRSB_OK;
}

#define SET_INPUT(name, MODE, STRIDE)                                                                        \
  int mrsb_set_input_##name(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload) {           \
    return mrsb_set_input(h, MODE, n, idx, payload, STRIDE);                                                 \
  }
SET_INPUT(actuators, MRSB_ACTUATOR_CMD, MRSB_MAX_MOTORS)
SET_INPUT(control_group, MRSB_CONTROL_GROUP_CMD, 4)
SET_INPUT(attitude_rate, MRSB_ATTITUDE_RATE_CMD, 4)
SET_INPUT(attitude, MRSB_ATTITUDE_CMD, 10)
SET_INPUT(tilt_hdg_rate, MRSB_TILT_HDG_RATE_CMD, 5)
SET_INPUT(acceleration_hdg_rate, MRSB_ACCELERATION_HDG_RATE_CMD, 4)
SET_INPUT(acceleration_hdg, MRSB_ACCELERATION_HDG_CMD, 4)
SET_INPUT(velocity_hdg_rate, MRSB_VELOCITY_HDG_RATE_CMD, 4)
SET_INPUT(velocity_hdg, MRSB_VELOCITY_HDG_CMD, 4)
SET_INPUT(position, MRSB_POSITION_CMD, 4)
#undef SET_INPUT

int mrsb_clear_input(mrsb_handle h, int64_t n, const int32_t* idx) {
  return mrsb_set_input(h, MRSB_INPUT_UNKNOWN, n, idx, nullptr, 0);
}

// host rows -> SoA rows [row0, row0+rows) of `dst`; then OR `flag` into the per-UAV flags
static int put_rows(mrsb_sim* h, double* dst, int rows_total, int row0, int rows, int64_t n, const int32_t* idx, const double* payload, int stride,
                    uint32_t or_flag) {
  const int32_t* d_idx  = nullptr;
  const double*  d_rows = nullptr;
  int            rc     = upload(h, n, idx, {{payload, stride}}, &d_idx, &d_rows);
  if (rc || n == 0) return rc;
  h->n_launches += launch_scatter_rows(dst, rows_total, row0, rows, n, d_idx, d_rows, stride, h->ds.perm, h->stream);
  if (or_flag) h->n_launches += launch_flag_update(h->ds, n, d_idx, 0xffffffffu, or_flag, h->stream);
  CU(cudaGetLastError());
  return MRSB_OK;
}

static int get_rows(mrsb_sim* h, const double* src, int rows_total, int row0, int rows, int64_t n, const int32_t* idx, double* out) {
  return download(h, n, idx, sizeof(double) * size_t(n) * size_t(rows), out, [&](const int32_t* d_idx, void* d_out) {
    return launch_gather_rows(src, rows_total, row0, rows, n, d_idx, static_cast<double*>(d_out), rows, h->ds.perm, h->stream);
  });
}

int mrsb_set_feedforward_acceleration_hdg_rate(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload) {
  GUARD(h);
  return put_rows(h, h->ds.ff, FF_ROWS, FF_ACC_HDG_RATE, 4, n, idx, payload, 4, FLAG_FF_ACC_HDG_RATE);
}
int mrsb_set_feedforward_acceleration_hdg(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload) {
  GUARD(h);
  return put_rows(h, h->ds.ff, FF_ROWS, FF_ACC_HDG, 3, n, idx, payload, 4, FLAG_FF_ACC_HDG);
}
int mrsb_set_feedforward_velocity_hdg(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload) {
  GUARD(h);
  return put_rows(h, h->ds.ff, FF_ROWS, FF_VEL_HDG, 3, n, idx, payload, 4, FLAG_FF_VEL_HDG);
}
int mrsb_set_feedforward_velocity_hdg_rate(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload) {
  GUARD(h);
  return put_rows(h, h->ds.ff, FF_ROWS, FF_VEL_HDG_RATE, 3, n, idx, payload, 4, FLAG_FF_VEL_HDG_RATE);
}
int mrsb_set_tracker_cmd(mrsb_handle h, int64_t n, const int32_t* idx, const double* rows) {
  GUARD(h);
  const int32_t* d_idx  = nullptr;
  const double*  d_rows = nullptr;
  int            rc     = upload(h, n, idx, {{rows, MRSB_TRACKER_CMD_STRIDE}}, &d_idx, &d_rows);  // validates n and idx before anything is read
  if (rc || n == 0) return rc;
  h->n_launches += launch_tracker_cmd(h->ds, n, d_idx, d_rows, h->stream);  // ROSW:995-1021 in one kernel
  CU(cudaGetLastError());
  return MRSB_OK;
}
int mrsb_clear_feedforward(mrsb_handle h, int64_t n, const int32_t* idx) {
  GUARD(h);
  const int32_t* d_idx = nullptr;
  int            rc    = stage_idx(h, n, idx, &d_idx);
  if (rc) return rc;
  h->n_launches += launch_flag_update(h->ds, n, d_idx, ~(FLAG_FF_ACC_HDG | FLAG_FF_ACC_HDG_RATE | FLAG_FF_VEL_HDG | FLAG_FF_VEL_HDG_RATE), 0u, h->stream);
  return MRSB_OK;
}

// ------------------------------------------------------------------------------------------
// stepping
// ------------------------------------------------------------------------------------------
static int exchange_positions(mrsb_sim* h) {
  if (h->n_ranks <= 1 || h->p2p) return MRSB_OK;  // pull exchange: nothing moves; the pass' first kernel hand-shakes
  if (!h->comm) return fail(MRSB_ERR_STATE, "sharded handle (n_global > n_local) without a communicator: call mrsb_comm_init_nccl, or use mrsb_gather_buffer + mrsb_handle_collisions_gathered");
  h->positions_touched = true;  // all-gather without the hand-shake: no swarm-wide displacement bound for this pass
  double* buf = h->ds.gpos;
  if (h->equal_shards) {
    NC(g_nccl.AllGather(buf + 3 * h->ds.shard_begin, buf, size_t(3 * h->ds.n), ncclDouble, h->comm, h->stream));
  } else {
    NC(g_nccl.GroupStart());
    for (int r = 0; r < h->n_ranks; r++) {
      double* p = buf + 3 * h->shard_begin_of[r];
      NC(g_nccl.Broadcast(p, p, size_t(3 * h->shard_count_of[r]), ncclDouble, r, h->comm, h->stream));
    }
    NC(g_nccl.GroupEnd());
  }
  return MRSB_OK;
}

// What the launches of the collision pass that comes next take (with_step: of a tick, its stepping launch first).  With the pull
// exchange, h->ds already points at the buffers of that pass' parity (after_pass).
static void graph_args(const mrsb_sim* h, bool with_step, double dt, int k_substeps, GraphArgs* a) {
  std::memset(static_cast<void*>(a), 0, sizeof(*a));  // padding included
  std::memcpy(&a->s, &h->ds, sizeof(DevState));
  std::memcpy(&a->grid, &h->grid, sizeof(DevGrid));
  std::memcpy(&a->pv, h->p2p ? &h->pv[write_buf(h)] : &h->pv_local, sizeof(PeerView));
  std::memcpy(&a->p2p, &h->p2pctl, sizeof(P2PCtl));
  a->crash = h->coll_crash, a->lists = h->lists_on, a->rebounce = h->coll_rebounce;
  if (!with_step) return;
  a->with_step = 1, a->k_substeps = k_substeps, a->uniform_mode = h->uniform_mode, a->any_moment = h->any_moment, a->dt = dt;
  a->publish   = h->p2p && h->ds.perm;  // bucketed: the per-group boxes follow the EXTERNAL order
  a->n_buckets = int(h->buckets.size());
  std::memcpy(a->buckets, h->buckets.data(), sizeof(Bucket) * h->buckets.size());
}

// the stepping launch: one kernel per bucket, each on its own view of the tiled arrays
static int launch_step_buckets(const GraphArgs& a, cudaStream_t stream, int* info) {
  int own = 0;
  for (int i = 0; i < a.n_buckets; i++) {
    const Bucket& b = a.buckets[i];
    if (b.count <= 0) continue;
    DevState v = a.s;
    if (b.slot0 > 0) {
      const int64_t t0 = b.slot0 / MRSB_TILE;
      v.st += t0 * ST_ROWS * MRSB_TILE, v.vprev += t0 * VPREV_ROWS * MRSB_TILE, v.rpm += t0 * MRSB_NM * MRSB_TILE, v.pid += t0 * PID_ROWS * MRSB_TILE;
      v.fext += t0 * F3_ROWS * MRSB_TILE, v.mext += t0 * F3_ROWS * MRSB_TILE, v.imu += t0 * F3_ROWS * MRSB_TILE, v.cmd += t0 * CMD_ROWS * MRSB_TILE;
      v.ff += t0 * FF_ROWS * MRSB_TILE, v.initz += b.slot0, v.flags += b.slot0, v.mode += b.slot0;
    }
    if (v.inv) {
      v.inv += b.slot0;
      v.gbox = nullptr;  // its warps are not the external 32-UAV groups: publish_positions_kernel writes the boxes (below)
    }
    v.n = b.count;
    own += launch_step(v, b.pset >= 0 ? &b.params : nullptr, a.dt, a.k_substeps, a.uniform_mode, b.nm, a.any_moment, stream, info);
  }
  if (a.publish) own += launch_publish_positions(a.s, stream);
  return own;
}

// decide -> IF (rebuild) { table, lists } -> check, captured into the graph being built on h->stream.
// The IF node's condition is set on the device by decide_kernel (cudaGraphSetConditional).
static bool capture_list_pass(mrsb_sim* h, const GraphArgs& a, cudaGraph_t graph, cudaStream_t* side, int* own_fixed, int* own_rebuild) {
  cudaStreamCaptureStatus status;
  const cudaGraphNode_t*  deps  = nullptr;
  size_t                  n_dep = 0;
  cudaGraphConditionalHandle handle;
  if (cudaGraphConditionalHandleCreate(&handle, graph, 0, cudaGraphCondAssignDefault) != cudaSuccess) return false;
  *own_fixed += launch_collide_decide(a.grid, a.p2p, 0, handle, 1, h->stream);
  if (cudaStreamGetCaptureInfo_v2(h->stream, &status, nullptr, &graph, &deps, &n_dep) != cudaSuccess) return false;
  cudaGraphNodeParams cp = {};
  cp.type                = cudaGraphNodeTypeConditional;
  cp.conditional.handle  = handle;
  cp.conditional.type    = cudaGraphCondTypeIf;
  cp.conditional.size    = 1;
  cudaGraphNode_t cond   = nullptr;
  if (cudaGraphAddNode(&cond, graph, deps, n_dep, &cp) != cudaSuccess) return false;
  cudaGraph_t body = cp.conditional.phGraph_out[0];
  if (!*side && cudaStreamCreateWithFlags(side, cudaStreamNonBlocking) != cudaSuccess) return false;
  if (cudaStreamBeginCaptureToGraph(*side, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal) != cudaSuccess) return false;
  *own_rebuild = launch_collide_rebuild(a.s, a.grid, a.pv, *side);
  *own_rebuild += launch_collide_check(a.s, a.grid, a.pv, a.crash, a.rebounce, 0, *side);  // the rebuilding pass' own list check
  cudaGraph_t body_out = nullptr;
  if (cudaStreamEndCapture(*side, &body_out) != cudaSuccess) return false;
  // The list check of an ordinary pass is captured BESIDE the conditional node (both depend on decide only): evaluating a
  // conditional node that is not taken takes ~10 us, which then overlaps the check instead of preceding it.  On a rebuilding
  // pass this launch returns at once (the body above ends with its own check).  The graph has two leaves; it is complete when
  // both are.
  *own_fixed += launch_collide_check(a.s, a.grid, a.pv, a.crash, a.rebounce, 1, h->stream);
  cudaGraphNode_t both[2] = {cond, nullptr};
  const cudaGraphNode_t* tail = nullptr;
  size_t                 n_tail = 0;
  if (cudaStreamGetCaptureInfo_v2(h->stream, &status, nullptr, &graph, &tail, &n_tail) != cudaSuccess || n_tail != 1) return false;
  both[1] = tail[0];
  if (cudaStreamUpdateCaptureDependencies(h->stream, both, 2, cudaStreamSetCaptureDependencies) != cudaSuccess) return false;
  return true;
}

// The graph of `a`: the stepping launch if a.with_step (mrsb_run's tick graph), then the pass with neighbour lists, or the full
// pass.  exec stays nullptr if the capture fails.
static Graph build_pass_graph(mrsb_sim* h, const GraphArgs& a) {
  Graph        g(a);
  cudaGraph_t  graph = nullptr;
  cudaStream_t side  = nullptr;
  bool         ok    = false;
  if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
    cudaGetLastError();
    return g;
  }
  do {
    cudaStreamCaptureStatus status;
    if (cudaStreamGetCaptureInfo_v2(h->stream, &status, nullptr, &graph, nullptr, nullptr) != cudaSuccess || !graph) break;
    if (a.with_step) g.own += launch_step_buckets(a, h->stream, h->step_info);
    if (a.lists) {
      ok = capture_list_pass(h, a, graph, &side, &g.own, &h->rebuild_own);
    } else {
      g.own += launch_collide(a.s, a.grid, a.pv, a.p2p, a.crash, a.rebounce, h->stream);
      ok = true;
    }
  } while (false);
  cudaGraph_t captured = nullptr;
  const bool  ended    = cudaStreamEndCapture(h->stream, &captured) == cudaSuccess && captured;
  if (ok && ended && cudaGraphInstantiate(&g.exec, captured, 0) != cudaSuccess) g.exec = nullptr;
  if (captured) cudaGraphDestroy(captured);
  if (side) cudaStreamDestroy(side);
  cudaGetLastError();
  return g;
}

// host bookkeeping before a pass that goes through decide_kernel
static int before_list_pass(mrsb_sim* h) {
  // anything but exactly one stepping launch since the last pass: the displacement bound does not cover it
  if (h->positions_touched || h->steps_since_pass != 1)
    CU(cudaMemcpyAsync(&h->grid.ctl->force, h->h_one.get(), sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  h->positions_touched = false;
  h->steps_since_pass  = 0;
  h->list_passes++;
  return MRSB_OK;
}

// host bookkeeping after any pass: with the pull exchange the write buffer changes sides
static int after_pass(mrsb_sim* h) {
  h->n_passes++;
  if (h->p2p) {
    h->pass_no++;
    const int w         = write_buf(h);
    h->ds.gpos          = h->gbuf[w];
    h->ds.gbox          = h->d_gbox[w];
    h->ds.geom          = h->d_geom[w];
    h->wrote_since_pass = false;
    int rc              = apply_pending_geom(h, w);  // no peer reads this buffer any more (they have all started the pass that just ran)
    if (rc) return rc;
  }
  CU(cudaGetLastError());
  return MRSB_OK;
}

static int collide_local(mrsb_sim* h) {
  if (h->p2p && !h->wrote_since_pass) {
    // nothing wrote positions since the last pass: the buffer this pass reads still holds the ones of two passes ago
    h->n_launches += launch_publish_positions(h->ds, h->stream);
    h->wrote_since_pass = true;
  }
  if (h->lists_on) {
    int rc = before_list_pass(h);
    if (rc) return rc;
  } else {
    h->steps_since_pass = 0;
  }
  GraphArgs a;
  graph_args(h, false, 0.0, 0, &a);
  Graph& g       = h->pass[write_buf(h)];
  bool   graphed = !h->graph_failed && !getenv("MRSB_NO_GRAPH");
  if (graphed && !(g.exec && g.holds(a))) {
    g               = build_pass_graph(h, a);
    graphed         = g.exec != nullptr;
    h->graph_failed = !graphed;
  }
  if (graphed) {
    CU(cudaGraphLaunch(g.exec, h->stream));
    h->n_launches += g.own;  // with neighbour lists the rebuilds are added from the device-side count (mrsb_get_counters)
  } else if (a.lists) {
    // no graph (MRSB_NO_GRAPH, or a capture failed): rebuild every pass
    h->n_launches += launch_collide_decide(a.grid, a.p2p, 1, cudaGraphConditionalHandle{}, 0, h->stream);
    h->rebuild_own = launch_collide_rebuild(a.s, a.grid, a.pv, h->stream);
    h->rebuild_own += launch_collide_check(a.s, a.grid, a.pv, a.crash, a.rebounce, 0, h->stream);
  } else {
    h->n_launches += launch_collide(a.s, a.grid, a.pv, a.p2p, a.crash, a.rebounce, h->stream);
  }
  return after_pass(h);
}

static int before_step(mrsb_sim* h, double dt, int32_t k_substeps) {
  if (k_substeps < 1) return fail(MRSB_ERR_INVALID, "k_substeps must be >= 1");
  int rc = flush_params(h);
  if (rc) return rc;
  rc = ensure_filt(h, dt);
  if (rc) return rc;
  if (h->p2p && *h->h_status.get()) return fail(MRSB_ERR_STATE, "peer hand-shake timed out (a rank stopped calling the collision pass)");
  return MRSB_OK;
}

int mrsb_make_step(mrsb_handle h, double dt, int32_t k_substeps) {
  GUARD(h);
  int rc = before_step(h, dt, k_substeps);
  if (rc) return rc;
  GraphArgs a;
  graph_args(h, true, dt, k_substeps, &a);
  h->n_launches += launch_step_buckets(a, h->stream, h->step_info);
  h->wrote_since_pass = true;
  h->n_steps += k_substeps;
  h->steps_since_pass++;
  CU(cudaGetLastError());
  return MRSB_OK;
}

static int before_collisions(mrsb_sim* h) {
  int rc = flush_params(h);
  if (rc) return rc;
  if (h->ds.n_global > h->ds.n && h->n_ranks <= 1) return fail(MRSB_ERR_STATE, "sharded handle without communicator");
  if (h->lists_on && (h->positions_touched || h->steps_since_pass != 1))
    // anything but exactly one stepping launch since the last pass: this rank's displacement is unbounded —
    // said through the displacement word, so that every peer rebuilds as well
    CU(cudaMemcpyAsync(&h->grid.ctl->disp_max_bits, h->h_one.get() + 1, sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  return MRSB_OK;
}

int mrsb_handle_collisions(mrsb_handle h) {
  GUARD(h);
  if (!(h->coll_crash || h->coll_enabled)) return MRSB_OK;  // SIM:299-301
  int rc = before_collisions(h);
  if (rc) return rc;
  rc = exchange_positions(h);
  if (rc) return rc;
  return collide_local(h);
}

int mrsb_handle_collisions_gathered(mrsb_handle h) {
  GUARD(h);
  if (!(h->coll_crash || h->coll_enabled)) return MRSB_OK;
  int rc = flush_params(h);
  if (rc) return rc;
  return collide_local(h);
}

// One tick = stepping launch + collision pass.  With neighbour lists the two are ONE graph (per buffer parity): a single
// cudaGraphLaunch per tick instead of a kernel launch plus a graph launch, and no gap between the stepping kernel and the
// pass' first kernel.
static int run_tick_graph(mrsb_sim* h, double dt, int32_t k_substeps, bool* done) {
  *done = false;
  if (!h->lists_on || h->graph_failed || getenv("MRSB_NO_GRAPH")) return MRSB_OK;
  if (h->positions_touched || h->steps_since_pass != 0) return MRSB_OK;  // let the ordinary path sort that out first
  GraphArgs a;
  graph_args(h, true, dt, k_substeps, &a);
  Graph& g = h->tick[write_buf(h)];
  if (!g.holds(a)) {
    g = Graph(a);
    return MRSB_OK;  // this tick goes the ordinary way (first launches set up function attributes: not inside a capture); the next one of this parity builds the graph
  }
  if (!g.exec) {
    g = build_pass_graph(h, a);
    if (!g.exec) {
      h->graph_failed = true;
      return MRSB_OK;
    }
  }
  // bookkeeping of make_step + before_collisions + collide_local for "exactly one stepping launch, then the pass"
  h->wrote_since_pass = true;
  h->n_steps += k_substeps;
  h->list_passes++;
  CU(cudaGraphLaunch(g.exec, h->stream));
  h->n_launches += g.own;
  *done = true;
  return after_pass(h);
}

int mrsb_run(mrsb_handle h, double dt, int32_t k_substeps, int32_t n_ticks, int32_t with_collisions) {
  GUARD(h);
  const bool collide = with_collisions && (h->coll_crash || h->coll_enabled);
  for (int t = 0; t < n_ticks; t++) {
    if (collide) {
      int rc = before_step(h, dt, k_substeps);
      if (rc) return rc;
      bool done = false;
      rc        = run_tick_graph(h, dt, k_substeps, &done);
      if (rc) return rc;
      if (done) continue;
    }
    int rc = mrsb_make_step(h, dt, k_substeps);
    if (rc) return rc;
    if (collide) {
      rc = mrsb_handle_collisions(h);
      if (rc) return rc;
    }
  }
  return MRSB_OK;
}

// ------------------------------------------------------------------------------------------
// state access
// ------------------------------------------------------------------------------------------
int mrsb_get_state(mrsb_handle h, int64_t n, const int32_t* idx, double* x, double* v, double* R, double* omega, double* motor_rpm) {
  GUARD(h);
  int rc = MRSB_OK;
  if (x && !rc) rc = get_rows(h, h->ds.st, ST_ROWS, 0, 3, n, idx, x);
  if (v && !rc) rc = get_rows(h, h->ds.st, ST_ROWS, 3, 3, n, idx, v);
  if (R && !rc) rc = get_rows(h, h->ds.st, ST_ROWS, 6, 9, n, idx, R);
  if (omega && !rc) rc = get_rows(h, h->ds.st, ST_ROWS, 15, 3, n, idx, omega);
  if (motor_rpm && !rc) rc = get_rows(h, h->ds.rpm, MRSB_NM, 0, MRSB_NM, n, idx, motor_rpm);
  return rc;
}

int mrsb_get_v_prev(mrsb_handle h, int64_t n, const int32_t* idx, double* v_prev) {
  GUARD(h);
  return download(h, n, idx, sizeof(double) * 3 * size_t(n), v_prev, [&](const int32_t* d_idx, void* d_out) {
    return launch_gather_vprev(h->ds, n, d_idx, static_cast<double*>(d_out), h->stream);
  });
}

int mrsb_get_imu_acceleration(mrsb_handle h, int64_t n, const int32_t* idx, double* acc) {
  GUARD(h);
  if (!(h->ds.opts & STEP_OPT_IMU)) return fail(MRSB_ERR_STATE, "the IMU rows are switched off (mrsb_set_outputs)");
  return get_rows(h, h->ds.imu, F3_ROWS, 0, 3, n, idx, acc);
}

int mrsb_set_state(mrsb_handle h, int64_t n, const int32_t* idx, const double* x, const double* v, const double* R, const double* omega,
                   const double* motor_rpm) {
  GUARD(h);
  int rc = MRSB_OK;
  if (v) {
    const int32_t* d_idx = nullptr;
    rc                   = stage_idx(h, n, idx, &d_idx);
    if (rc) return rc;
    h->n_launches += launch_stash_vprev(h->ds, n, d_idx, h->stream);
  }
  if (x && !rc) rc = put_rows(h, h->ds.st, ST_ROWS, 0, 3, n, idx, x, 3, 0);
  if (v && !rc) rc = put_rows(h, h->ds.st, ST_ROWS, 3, 3, n, idx, v, 3, 0);
  if (R && !rc) rc = put_rows(h, h->ds.st, ST_ROWS, 6, 9, n, idx, R, 9, 0);
  if (omega && !rc) rc = put_rows(h, h->ds.st, ST_ROWS, 15, 3, n, idx, omega, 3, 0);
  if (motor_rpm && !rc) rc = put_rows(h, h->ds.rpm, MRSB_NM, 0, MRSB_NM, n, idx, motor_rpm, MRSB_NM, 0);
  if (x && !rc) {
    h->n_launches += launch_publish_positions(h->ds, h->stream);
    h->wrote_since_pass  = true;
    h->positions_touched = true;
  }
  return rc;
}

int mrsb_set_state_pos(mrsb_handle h, int64_t n, const int32_t* idx, const double* xyz, const double* heading) {
  GUARD(h);
  const int32_t* d_idx = nullptr;
  const double*  d[2]  = {nullptr, nullptr};  // xyz, heading
  int            rc    = upload(h, n, idx, {{xyz, 3}, {heading, 1}}, &d_idx, d);
  if (rc || n == 0) return rc;
  h->n_launches += launch_set_state_pos(h->ds, n, d_idx, d[0], d[1], h->stream);
  if (h->p2p) h->n_launches += launch_publish_positions(h->ds, h->stream);  // the whole slice of the buffer being written, and its group boxes
  h->wrote_since_pass  = true;
  h->positions_touched = true;
  CU(cudaGetLastError());
  return MRSB_OK;
}

// The next pass that goes through decide_kernel replaces every force it visits (SIM:356-358), not only the ones it knows to be
// non-zero.  No host synchronisation: the copy reads the pinned word when it runs.  If a later call has raised the word by then,
// more passes than needed write every force they visit, which writes the values they would have left in place.
static int write_all_forces_next_pass(mrsb_sim* h) {
  if (!h->grid.ctl) return MRSB_OK;
  *h->h_until.get() = (unsigned long long)h->list_passes + 1ull;  // index of the next pass that goes through decide_kernel
  CU(cudaMemcpyAsync(&h->grid.ctl->write_all_until, h->h_until.get(), sizeof(unsigned long long), cudaMemcpyHostToDevice, h->stream));
  return MRSB_OK;
}

// forces were written by something else than the collision pass: the next pass must replace every UAV's force
static int forces_written(mrsb_sim* h) {
  int rc = write_all_forces_next_pass(h);
  if (rc) return rc;
  h->positions_touched = true;  // that pass rebuilds: UAVs without candidates are only visited by a rebuild
  return MRSB_OK;
}

// after a respawn: the buffer peers read has to show the new positions, and their per-group boxes (pull exchange)
static int respawned(mrsb_sim* h) {
  if (h->p2p) h->n_launches += launch_publish_positions(h->ds, h->stream);
  h->wrote_since_pass = true;
  CU(cudaGetLastError());
  return MRSB_OK;
}

int mrsb_respawn(mrsb_handle h, int64_t n, const int32_t* idx, const double* xyz, const double* heading) {
  GUARD(h);
  const int32_t* d_idx = nullptr;
  const double*  d[2]  = {nullptr, nullptr};  // xyz, heading
  int            rc    = upload(h, n, idx, {{xyz, 3}, {heading, 1}}, &d_idx, d);
  if (rc || n == 0) return rc;
  rc = flush_params(h);  // the kernel reads the take-off flag of every UAV's parameter set
  if (rc) return rc;
  h->n_launches += launch_respawn(h->ds, h->d_takeoff0.get(), n, d_idx, d[0], d[1], h->stream);
  h->positions_touched = true;
  note_mode(h, MRSB_INPUT_UNKNOWN, n, idx == nullptr);
  return respawned(h);
}

int mrsb_respawn_masked_device(mrsb_handle h, const uint8_t* mask_dev, const double* xyz_dev, const double* heading_dev) {
  GUARD(h);
  if (!mask_dev || !xyz_dev || !heading_dev) return fail(MRSB_ERR_INVALID, "null device pointer");
  int rc = flush_params(h);
  if (rc) return rc;
  // the host does not learn who was respawned: the kernel raises the displacement word itself (no forced rebuild from here), and
  // the batch can no longer be assumed to share one input mode unless it is already INPUT_UNKNOWN
  h->n_launches += launch_respawn_masked(h->ds, h->d_takeoff0.get(), mask_dev, xyz_dev, heading_dev, h->stream);
  note_mode(h, MRSB_INPUT_UNKNOWN, 1, false);
  return respawned(h);
}

// ---- snapshots ------------------------------------------------------------------------------
static size_t snapshot_bytes(const mrsb_sim* h) {
  return size_t(h->ds.n) * (sizeof(double) * SNAP_ROWS + sizeof(uint32_t) + sizeof(uint8_t));
}

// the snapshot `id` of this handle, or nullptr (and MRSB_ERR_INVALID in *rc)
static mrsb_sim::Snapshot* find_snapshot(mrsb_sim* h, int32_t id, int* rc) {
  auto it = h->snapshots.find(id);
  if (it != h->snapshots.end()) return &it->second;
  *rc = fail(MRSB_ERR_INVALID, "no snapshot %d on this handle", id);
  return nullptr;
}

struct SnapshotParts {
  double*   rows;
  uint32_t* flags;
  uint8_t*  mode;
};
static SnapshotParts parts_of(const mrsb_sim* h, mrsb_sim::Snapshot& s) {
  const size_t n = size_t(h->ds.n);
  double*      r = reinterpret_cast<double*>(s.mem.get());
  uint32_t*    f = reinterpret_cast<uint32_t*>(r + SNAP_ROWS * n);
  return {r, f, reinterpret_cast<uint8_t*>(f + n)};
}

// The header of a snapshot image; the snapshot's device bytes follow it verbatim.
struct SnapshotImageHeader {
  char     magic[8];  // "MRSBSNAP"
  uint32_t version, rows;
  int64_t  n_local, n_global, shard_begin;
  int32_t  uniform_mode, any_moment;
};
static const char     kSnapshotMagic[8]  = {'M', 'R', 'S', 'B', 'S', 'N', 'A', 'P'};
static const uint32_t kSnapshotVersion = 1;

int mrsb_snapshot_create(mrsb_handle h, int32_t* id) {
  GUARD(h);
  if (!id) return fail(MRSB_ERR_INVALID, "null id");
  mrsb_sim::Snapshot s;
  int rc = s.mem.alloc(std::max<size_t>(snapshot_bytes(h), 1));
  if (rc) return rc;
  *id = h->next_snapshot++;
  h->snapshots.emplace(*id, std::move(s));
  return MRSB_OK;
}

int mrsb_snapshot_free(mrsb_handle h, int32_t id) {
  GUARD(h);
  int rc = MRSB_OK;
  if (!find_snapshot(h, id, &rc)) return rc;
  CU(cudaStreamSynchronize(h->stream));  // a save or restore may still read or write it
  h->snapshots.erase(id);
  return MRSB_OK;
}

int mrsb_snapshot_save(mrsb_handle h, int32_t id) {
  GUARD(h);
  int                 rc = MRSB_OK;
  mrsb_sim::Snapshot* s  = find_snapshot(h, id, &rc);
  if (!s) return rc;
  const SnapshotParts p = parts_of(h, *s);
  h->n_launches += launch_snapshot_save(h->ds, p.rows, p.flags, p.mode, h->stream);
  s->filled       = true;
  s->uniform_mode = h->uniform_mode;
  s->any_moment   = h->any_moment;
  CU(cudaGetLastError());
  return MRSB_OK;
}

// host bookkeeping after a restore.  all_own: every UAV took its own record.
static int restored(mrsb_sim* h, const mrsb_sim::Snapshot& s, bool all_own) {
  h->any_moment   = h->any_moment || s.any_moment;
  h->uniform_mode = (all_own || h->uniform_mode == s.uniform_mode) ? s.uniform_mode : -1;
  return respawned(h);
}

int mrsb_snapshot_restore(mrsb_handle h, int32_t id, int64_t n, const int32_t* idx, const int32_t* src) {
  GUARD(h);
  int                 rc = MRSB_OK;
  mrsb_sim::Snapshot* s  = find_snapshot(h, id, &rc);
  if (!s) return rc;
  if (!s->filled) return fail(MRSB_ERR_STATE, "snapshot %d was never saved or uploaded", id);
  const int32_t* d_idx = nullptr;
  rc                   = stage_idx(h, n, idx, &d_idx);
  if (rc || n == 0) return rc;
  const int32_t* d_src = nullptr;
  if (src) {
    for (int64_t k = 0; k < n; k++)
      if (src[k] < 0 || src[k] >= h->ds.n) return fail(MRSB_ERR_INVALID, "src[%lld]=%d outside 0..%lld", (long long)k, src[k], (long long)h->ds.n - 1);
    rc = ensure_stage(h, sizeof(int32_t) * size_t(n));
    if (rc) return rc;
    CU(cudaMemcpyAsync(h->d_stage.get(), src, sizeof(int32_t) * size_t(n), cudaMemcpyHostToDevice, h->stream));
    d_src = reinterpret_cast<const int32_t*>(h->d_stage.get());
  }
  rc = forces_written(h);  // a restored external force may be non-zero where the next list-only pass would not look
  if (rc) return rc;
  const SnapshotParts p = parts_of(h, *s);
  h->n_launches += launch_snapshot_restore(h->ds, p.rows, p.flags, p.mode, n, d_idx, d_src, h->stream);
  h->positions_touched = true;
  return restored(h, *s, !idx && !src && n == h->ds.n);
}

int mrsb_snapshot_restore_device(mrsb_handle h, int32_t id, const int32_t* src_dev) {
  GUARD(h);
  int                 rc = MRSB_OK;
  mrsb_sim::Snapshot* s  = find_snapshot(h, id, &rc);
  if (!s) return rc;
  if (!s->filled) return fail(MRSB_ERR_STATE, "snapshot %d was never saved or uploaded", id);
  // the host does not learn who was restored: the kernel raises the displacement word itself (the next pass rebuilds only if
  // somebody was), and the next pass that goes through decide_kernel writes every force it visits
  rc = write_all_forces_next_pass(h);
  if (rc) return rc;
  const SnapshotParts p = parts_of(h, *s);
  h->n_launches += launch_snapshot_restore_masked(h->ds, p.rows, p.flags, p.mode, src_dev, h->stream);
  return restored(h, *s, src_dev == nullptr);
}

int mrsb_snapshot_image_size(mrsb_handle h, size_t* bytes) {
  GUARD(h);
  if (!bytes) return fail(MRSB_ERR_INVALID, "null output");
  *bytes = sizeof(SnapshotImageHeader) + snapshot_bytes(h);
  return MRSB_OK;
}

int mrsb_snapshot_download(mrsb_handle h, int32_t id, void* host, size_t bytes) {
  GUARD(h);
  int                 rc = MRSB_OK;
  mrsb_sim::Snapshot* s  = find_snapshot(h, id, &rc);
  if (!s) return rc;
  if (!host || bytes != sizeof(SnapshotImageHeader) + snapshot_bytes(h))
    return fail(MRSB_ERR_INVALID, "image buffer of %zu bytes, need %zu (mrsb_snapshot_image_size)", bytes, sizeof(SnapshotImageHeader) + snapshot_bytes(h));
  if (!s->filled) return fail(MRSB_ERR_STATE, "snapshot %d was never saved or uploaded", id);
  SnapshotImageHeader hd;
  std::memset(&hd, 0, sizeof(hd));
  std::memcpy(hd.magic, kSnapshotMagic, sizeof(hd.magic));
  hd.version = kSnapshotVersion, hd.rows = SNAP_ROWS;
  hd.n_local = h->ds.n, hd.n_global = h->ds.n_global, hd.shard_begin = h->ds.shard_begin;
  hd.uniform_mode = s->uniform_mode, hd.any_moment = s->any_moment ? 1 : 0;
  std::memcpy(host, &hd, sizeof(hd));
  if (h->ds.n) CU(cudaMemcpyAsync(static_cast<char*>(host) + sizeof(hd), s->mem.get(), snapshot_bytes(h), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return MRSB_OK;
}

int mrsb_snapshot_upload(mrsb_handle h, int32_t id, const void* host, size_t bytes) {
  GUARD(h);
  int                 rc = MRSB_OK;
  mrsb_sim::Snapshot* s  = find_snapshot(h, id, &rc);
  if (!s) return rc;
  if (!host || bytes != sizeof(SnapshotImageHeader) + snapshot_bytes(h))
    return fail(MRSB_ERR_INVALID, "image of %zu bytes, this handle's are %zu", bytes, sizeof(SnapshotImageHeader) + snapshot_bytes(h));
  SnapshotImageHeader hd;
  std::memcpy(&hd, host, sizeof(hd));
  if (std::memcmp(hd.magic, kSnapshotMagic, sizeof(hd.magic)) != 0 || hd.version != kSnapshotVersion || hd.rows != SNAP_ROWS)
    return fail(MRSB_ERR_INVALID, "not a snapshot image of this library version");
  if (hd.n_local != h->ds.n || hd.n_global != h->ds.n_global || hd.shard_begin != h->ds.shard_begin)
    return fail(MRSB_ERR_INVALID, "image of a shard of %lld UAVs at %lld of %lld, this handle has %lld at %lld of %lld", (long long)hd.n_local,
                (long long)hd.shard_begin, (long long)hd.n_global, (long long)h->ds.n, (long long)h->ds.shard_begin, (long long)h->ds.n_global);
  if (hd.uniform_mode < -1 || hd.uniform_mode > MRSB_POSITION_CMD || (hd.any_moment != 0 && hd.any_moment != 1))
    return fail(MRSB_ERR_INVALID, "corrupt snapshot image header");
  if (h->ds.n) CU(cudaMemcpyAsync(s->mem.get(), static_cast<const char*>(host) + sizeof(hd), snapshot_bytes(h), cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));  // the caller may release `host` on return
  s->filled       = true;
  s->uniform_mode = hd.uniform_mode;
  s->any_moment   = hd.any_moment != 0;
  return MRSB_OK;
}

int mrsb_get_input_mode(mrsb_handle h, int64_t n, const int32_t* idx, int32_t* mode) {
  GUARD(h);
  return download(h, n, idx, sizeof(int32_t) * size_t(n), mode, [&](const int32_t* d_idx, void* d_out) {
    return launch_gather_u8(h->ds.mode, n, d_idx, static_cast<int32_t*>(d_out), h->ds.perm, h->stream);
  });
}

static int get_flags(mrsb_sim* h, int64_t n, const int32_t* idx, uint32_t* out) {
  return download(h, n, idx, sizeof(uint32_t) * size_t(n), out, [&](const int32_t* d_idx, void* d_out) {
    return launch_gather_u32(h->ds.flags, n, d_idx, static_cast<uint32_t*>(d_out), h->ds.perm, h->stream);
  });
}

int mrsb_crash(mrsb_handle h, int64_t n, const int32_t* idx) {
  GUARD(h);
  const int32_t* d_idx = nullptr;
  int            rc    = stage_idx(h, n, idx, &d_idx);
  if (rc) return rc;
  h->n_launches += launch_flag_update(h->ds, n, d_idx, 0xffffffffu, FLAG_CRASHED, h->stream);
  return MRSB_OK;
}

int mrsb_has_crashed(mrsb_handle h, int64_t n, const int32_t* idx, int32_t* crashed) {
  GUARD(h);
  int rc = get_flags(h, n, idx, reinterpret_cast<uint32_t*>(crashed));  // the flags, then in place what they say
  if (rc) return rc;
  for (int64_t k = 0; k < n; k++) crashed[k] = (uint32_t(crashed[k]) & FLAG_CRASHED) ? 1 : 0;
  return MRSB_OK;
}

int mrsb_forces_written(mrsb_handle h) {
  GUARD(h);
  return forces_written(h);
}

int mrsb_apply_force(mrsb_handle h, int64_t n, const int32_t* idx, const double* force) {
  GUARD(h);
  int rc = forces_written(h);
  if (rc) return rc;
  return put_rows(h, h->ds.fext, F3_ROWS, 0, 3, n, idx, force, 3, 0);
}
int mrsb_get_external_force(mrsb_handle h, int64_t n, const int32_t* idx, double* force) {
  GUARD(h);
  return get_rows(h, h->ds.fext, F3_ROWS, 0, 3, n, idx, force);
}
int mrsb_set_external_moment(mrsb_handle h, int64_t n, const int32_t* idx, const double* moment) {
  GUARD(h);
  h->any_moment = true;
  return put_rows(h, h->ds.mext, F3_ROWS, 0, 3, n, idx, moment, 3, 0);
}

// ------------------------------------------------------------------------------------------
// parameters
// ------------------------------------------------------------------------------------------
static int check_uav(mrsb_sim* h, int64_t uav) {
  if (uav < 0 || uav >= h->ds.n) return fail(MRSB_ERR_INVALID, "uav %lld outside 0..%lld", (long long)uav, (long long)h->ds.n - 1);
  return MRSB_OK;
}

int mrsb_get_params(mrsb_handle h, int64_t uav, mrsb_model_params* out) {
  GUARD(h);
  int rc = check_uav(h, uav);
  if (rc) return rc;
  *out = h->sets[h->pset_host[size_t(h->ds.shard_begin + uav)]].mp;
  uint32_t      fl  = 0;
  const int32_t one = int32_t(uav);
  rc                = get_flags(h, 1, &one, &fl);
  if (rc) return rc;
  out->takeoff_patch_enabled = (fl & FLAG_TAKEOFF) ? 1 : 0;
  return MRSB_OK;
}

int mrsb_get_controller_params(mrsb_handle h, int64_t uav, mrsb_controller_params* out) {
  GUARD(h);
  int rc = check_uav(h, uav);
  if (rc) return rc;
  *out = h->sets[h->pset_host[size_t(h->ds.shard_begin + uav)]].cp;
  return MRSB_OK;
}

int mrsb_get_mixer_allocation(mrsb_handle h, int64_t uav, double* out) {
  GUARD(h);
  int rc = check_uav(h, uav);
  if (rc) return rc;
  double mix[MRSB_MAX_MOTORS][4];
  mrsb_mixer_allocation(h->sets[h->pset_host[size_t(h->ds.shard_begin + uav)]].mp, mix);
  std::memcpy(out, mix, sizeof(mix));
  return MRSB_OK;
}

int mrsb_set_params(mrsb_handle h, int64_t n, const int32_t* idx, const mrsb_model_params* params) {
  GUARD(h);
  if (!params) return fail(MRSB_ERR_INVALID, "null params");
  int rc = check_params(*params);
  if (rc) return rc;
  mrsb_controller_params def;
  mrsb_controller_params_default(&def);
  rc = repoint(h, n, idx, [&](ParamSet& s, int64_t) {  // US:404-409: new model params, controllers re-created with default gains
    s.mp = *params;
    s.cp = def;
  }, [](int64_t) { return uint64_t(0); });
  if (rc) return rc;
  const int32_t* d_idx = nullptr;
  rc                   = stage_idx(h, n, idx, &d_idx);
  if (rc) return rc;
  h->n_launches += launch_reset_pid(h->ds, n, d_idx, 0, 12, h->stream);
  h->n_launches += launch_flag_update(h->ds, n, d_idx, ~FLAG_TAKEOFF, params->takeoff_patch_enabled ? FLAG_TAKEOFF : 0u, h->stream);
  return MRSB_OK;
}

static int set_ctrl(mrsb_sim* h, int64_t n, const int32_t* idx, int pid_row0, int pid_rows, void (*edit)(ParamSet&, const double*), const double* v) {
  int rc = repoint(h, n, idx, [&](ParamSet& s, int64_t) { edit(s, v); }, [](int64_t) { return uint64_t(0); });
  if (rc) return rc;
  if (pid_rows) {
    const int32_t* d_idx = nullptr;
    rc                   = stage_idx(h, n, idx, &d_idx);
    if (rc) return rc;
    h->n_launches += launch_reset_pid(h->ds, n, d_idx, pid_row0, pid_rows, h->stream);
  }
  return MRSB_OK;
}

int mrsb_set_mixer_params(mrsb_handle h, int64_t n, const int32_t* idx, int32_t desaturation) {
  GUARD(h);
  const double v[1] = {double(desaturation)};
  return set_ctrl(h, n, idx, 0, 0, [](ParamSet& s, const double* v) { s.cp.mixer_desaturation = v[0] != 0.0; }, v);
}
int mrsb_set_rate_controller_params(mrsb_handle h, int64_t n, const int32_t* idx, double kp, double kd, double ki) {
  GUARD(h);
  const double v[3] = {kp, kd, ki};
  return set_ctrl(h, n, idx, 9, 3, [](ParamSet& s, const double* v) { s.cp.rate_kp = v[0], s.cp.rate_kd = v[1], s.cp.rate_ki = v[2]; }, v);
}
int mrsb_set_attitude_controller_params(mrsb_handle h, int64_t n, const int32_t* idx, double kp, double kd, double ki, double max_rate_roll_pitch,
                                        double max_rate_yaw) {
  GUARD(h);
  const double v[5] = {kp, kd, ki, max_rate_roll_pitch, max_rate_yaw};
  return set_ctrl(h, n, idx, 6, 3, [](ParamSet& s, const double* v) {
    s.cp.att_kp = v[0], s.cp.att_kd = v[1], s.cp.att_ki = v[2], s.cp.att_max_rate_roll_pitch = v[3], s.cp.att_max_rate_yaw = v[4];
  }, v);
}
int mrsb_set_velocity_controller_params(mrsb_handle h, int64_t n, const int32_t* idx, double kp, double kd, double ki, double max_acceleration) {
  GUARD(h);
  const double v[4] = {kp, kd, ki, max_acceleration};
  return set_ctrl(h, n, idx, 3, 3, [](ParamSet& s, const double* v) {
    s.cp.vel_kp = v[0], s.cp.vel_kd = v[1], s.cp.vel_ki = v[2], s.cp.vel_max_acceleration = v[3];
  }, v);
}
int mrsb_set_position_controller_params(mrsb_handle h, int64_t n, const int32_t* idx, double kp, double kd, double ki, double max_velocity) {
  GUARD(h);
  const double v[4] = {kp, kd, ki, max_velocity};
  return set_ctrl(h, n, idx, 0, 3, [](ParamSet& s, const double* v) {
    s.cp.pos_kp = v[0], s.cp.pos_kd = v[1], s.cp.pos_ki = v[2], s.cp.pos_max_velocity = v[3];
  }, v);
}

// ------------------------------------------------------------------------------------------
// ROS-wrapper arithmetic around the path
// ------------------------------------------------------------------------------------------
int mrsb_timeout_input(mrsb_handle h, int64_t n, const int32_t* idx) {
  GUARD(h);
  const int32_t* d_idx = nullptr;
  int            rc    = stage_idx(h, n, idx, &d_idx);
  if (rc) return rc;
  h->n_launches += launch_timeout_input(h->ds, n, d_idx, h->stream);
  CU(cudaGetLastError());
  return MRSB_OK;
}

static int observe(mrsb_sim* h, int what, int width, int64_t n, const int32_t* idx, double* out) {
  if (!out) return fail(MRSB_ERR_INVALID, "null output");
  if ((what == 1 || what == 3) && !(h->ds.opts & STEP_OPT_IMU)) return fail(MRSB_ERR_STATE, "the IMU rows are switched off (mrsb_set_outputs)");
  int rc = flush_params(h);
  if (rc) return rc;
  return download(h, n, idx, sizeof(double) * size_t(n) * size_t(width), out, [&](const int32_t* d_idx, void* d_out) {
    return launch_observe(h->ds, what, n, d_idx, static_cast<double*>(d_out), width, h->stream);
  });
}
int mrsb_get_odometry(mrsb_handle h, int64_t n, const int32_t* idx, double* out13) {
  GUARD(h);
  return observe(h, 0, 13, n, idx, out13);
}
int mrsb_get_imu(mrsb_handle h, int64_t n, const int32_t* idx, double* out10) {
  GUARD(h);
  return observe(h, 1, 10, n, idx, out10);
}
int mrsb_get_rangefinder(mrsb_handle h, int64_t n, const int32_t* idx, double* out1) {
  GUARD(h);
  return observe(h, 2, 1, n, idx, out1);
}
int mrsb_pack_observations_device(mrsb_handle h, double* out_dev, int32_t stride) {
  GUARD(h);
  if (!out_dev || stride < 17) return fail(MRSB_ERR_INVALID, "need a device buffer with rows of >= 17 doubles");
  if (!(h->ds.opts & STEP_OPT_IMU)) return fail(MRSB_ERR_STATE, "the IMU rows are switched off (mrsb_set_outputs)");
  int rc = flush_params(h);
  if (rc) return rc;
  h->n_launches += launch_observe(h->ds, 3, h->ds.n, nullptr, out_dev, stride, h->stream);
  CU(cudaGetLastError());
  return MRSB_OK;
}

// The neighbour table's workspace for this handle's n_local UAVs: >= 1.5 buckets per UAV, as the collision table.
static int grow_neighbour_table(mrsb_sim* h, DevGrid* t) {
  const size_t n    = size_t(h->ds.n);
  uint32_t     bits = 10;
  while (2 * (size_t(1) << bits) < 3 * n && bits < 30) bits++;
  t->n_buckets        = 1u << bits;
  t->scan_tiles       = scan_tiles_for(int64_t(t->n_buckets) + 3);
  auto&        w      = h->nb;
  const size_t nbk    = size_t(t->n_buckets) + 4;  // + mirrors of buckets 0 and 1 + sentinel
  int          rc     = w.pos.grow(3 * n, 3 * n, h->stream);
  if (!rc) rc = w.vel.grow(3 * n, 3 * n, h->stream);
  if (!rc) rc = w.bucket.grow(n, n, h->stream);
  if (!rc) rc = w.rank.grow(n, n, h->stream);
  if (!rc) rc = w.count.grow(nbk, nbk, h->stream);
  if (!rc) rc = w.begin.grow(nbk, nbk, h->stream);
  if (!rc) rc = w.rec.grow(2 * n, 2 * n, h->stream);  // worst case: every UAV in bucket 0 and mirrored
  if (!rc) rc = w.scan.grow(size_t(t->scan_tiles) + 1, size_t(t->scan_tiles) + 1, h->stream);
  if (rc) return rc;
  t->bucket = w.bucket.get(), t->rank = w.rank.get(), t->count = w.count.get(), t->begin = w.begin.get();
  t->rec = w.rec.get(), t->scan_state = w.scan.get();
  return MRSB_OK;
}

int mrsb_pack_neighbours_device(mrsb_handle h, double radius, int32_t k, int32_t* idx_dev, double* rows_dev, int32_t stride, int32_t* count_dev) {
  GUARD(h);
  if (!idx_dev && !rows_dev && !count_dev) return fail(MRSB_ERR_INVALID, "all outputs are NULL");
  if (!std::isfinite(radius) || !(radius > 0.0)) return fail(MRSB_ERR_INVALID, "radius=%g is not a finite positive number", radius);
  if (k < 1 || k > MRSB_MAX_NEIGHBOURS) return fail(MRSB_ERR_INVALID, "k=%d outside 1..%d", k, MRSB_MAX_NEIGHBOURS);
  if (rows_dev && stride < 6 * k) return fail(MRSB_ERR_INVALID, "stride=%d below 6*k=%d", stride, 6 * k);
  if (h->ds.n_global > h->ds.n) return fail(MRSB_ERR_STATE, "neighbour observations of a sharded handle (n_global > n_local) are not supported");
  if (h->ds.n <= 0) return MRSB_OK;
  DevGrid t{};
  int     rc = grow_neighbour_table(h, &t);
  if (rc) return rc;
  // The stencil covers [q - reach, q + reach) per axis.  A neighbour differs from q by less than radius * (1 + 2^-51) per axis
  // (rounding of d2 and of radius * radius), and the rounding of q - reach and of v * inv_cell moves a cell boundary by at most
  // 3 * 2^-53 * |v| in length: a relative margin of 2^-20 covers both for |coordinates| <= 2^30 * radius.
  t.reach    = radius * (1.0 + 0x1p-20);
  t.inv_cell = 1.0 / (2.0 * t.reach);  // the collision pass' layout: 2 x 2 stencil rows of 2 cells
  h->n_launches += launch_neighbours(h->ds, t, h->nb.pos.get(), h->nb.vel.get(), radius * radius, k, idx_dev, rows_dev, stride, count_dev, h->stream);
  CU(cudaGetLastError());
  return MRSB_OK;
}

// set_mass / set_ground_z services: getParams -> edit -> setParams for every addressed UAV (ROSW:1028-1080), as ONE batched
// re-pointing: UAVs that share the old parameter set and the new value share the new set; setParams' side effects (controllers
// back to default gains, PIDs reset, US:404-409) are applied with one launch each.  The take-off patch flag is the UAV's live
// one (getParams returns it, MM:275), so it does not change.
static int edit_params_each(mrsb_sim* h, int64_t n, const int32_t* idx, const double* value, void (*edit)(mrsb_model_params&, double)) {
  if (n < 0 || (!idx && n > h->ds.n)) return fail(MRSB_ERR_INVALID, "n=%lld outside 0..%lld", (long long)n, (long long)h->ds.n);
  mrsb_controller_params def;
  mrsb_controller_params_default(&def);
  int rc = repoint(h, n, idx, [&](ParamSet& s, int64_t k) {
    edit(s.mp, value[k]);
    s.cp = def;
  }, [&](int64_t k) {
    uint64_t bits;
    std::memcpy(&bits, &value[k], sizeof(bits));
    return bits;
  });
  if (rc) return rc;
  const int32_t* d_idx = nullptr;
  rc                   = stage_idx(h, n, idx, &d_idx);
  if (rc) return rc;
  h->n_launches += launch_reset_pid(h->ds, n, d_idx, 0, 12, h->stream);
  CU(cudaGetLastError());
  return MRSB_OK;
}

int mrsb_set_mass(mrsb_handle h, int64_t n, const int32_t* idx, const double* mass) {
  GUARD(h);
  if (!mass && n) return fail(MRSB_ERR_INVALID, "null mass");
  return edit_params_each(h, n, idx, mass, [](mrsb_model_params& p, double m) {
    const double original = p.mass;
    p.mass                = m;
    for (int k = 0; k < p.n_motors; k++)
      p.allocation_matrix[2 * MRSB_MAX_MOTORS + k] = p.mass * (p.allocation_matrix[2 * MRSB_MAX_MOTORS + k] / original);
    std::memset(p.J, 0, sizeof(p.J));
    p.J[0] = p.mass * (3.0 * p.arm_length * p.arm_length + p.body_height * p.body_height) / 12.0;
    p.J[4] = p.mass * (3.0 * p.arm_length * p.arm_length + p.body_height * p.body_height) / 12.0;
    p.J[8] = (p.mass * p.arm_length * p.arm_length) / 2.0;
  });
}

int mrsb_set_ground_z(mrsb_handle h, int64_t n, const int32_t* idx, const double* ground_z) {
  GUARD(h);
  if (!ground_z && n) return fail(MRSB_ERR_INVALID, "null ground_z");
  return edit_params_each(h, n, idx, ground_z, [](mrsb_model_params& p, double z) { p.ground_z = z; });
}

// ------------------------------------------------------------------------------------------
// collisions
// ------------------------------------------------------------------------------------------
// which optional rows the stepping kernel stores: the caller's wishes plus what the library itself needs
static int refresh_opts(mrsb_sim* h) {
  const bool     need_pos = (h->outputs & MRSB_OUT_POSITIONS) || h->coll_enabled || h->coll_crash || h->ds.n_global > h->ds.n;
  const uint32_t opts     = ((h->outputs & MRSB_OUT_IMU) ? STEP_OPT_IMU : 0u) | (need_pos ? STEP_OPT_GPOS : 0u) | (h->iterate_without_input ? 0u : STEP_OPT_NEED_INPUT);
  if (opts == h->ds.opts) return MRSB_OK;
  const bool pos_back = (opts & STEP_OPT_GPOS) && !(h->ds.opts & STEP_OPT_GPOS);
  h->ds.opts          = opts;
  if (pos_back) {  // the packed positions were not kept up to date meanwhile
    h->n_launches += launch_publish_positions(h->ds, h->stream);
    h->wrote_since_pass  = true;
    h->positions_touched = true;
    CU(cudaGetLastError());
  }
  return MRSB_OK;
}

int mrsb_set_collisions(mrsb_handle h, int32_t enabled, int32_t crash, double rebounce) {
  GUARD(h);
  h->coll_enabled  = enabled != 0;
  h->coll_crash    = crash != 0;
  h->coll_rebounce = rebounce;
  return refresh_opts(h);
}

int mrsb_set_outputs(mrsb_handle h, uint32_t mask) {
  GUARD(h);
  h->outputs = mask;
  return refresh_opts(h);
}

int mrsb_set_iterate_without_input(mrsb_handle h, int32_t enabled) {
  GUARD(h);
  h->iterate_without_input = enabled != 0;
  return refresh_opts(h);
}

int mrsb_get_collision_pairs(mrsb_handle h, int32_t* ij, int64_t cap, int64_t* count) {
  GUARD(h);
  unsigned long long found = 0;
  CU(cudaMemcpyAsync(&found, h->grid.counters, sizeof(found), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  if (count) *count = int64_t(found);
  if (int64_t(found) > h->grid.pair_cap)
    return fail(MRSB_ERR_CAPACITY, "%llu pairs found but the device pair buffer holds %lld", found, (long long)h->grid.pair_cap);
  if (!ij || found == 0) return MRSB_OK;
  std::vector<int32_t> tmp(2 * size_t(found));
  CU(cudaMemcpy(tmp.data(), h->grid.pairs, sizeof(int32_t) * tmp.size(), cudaMemcpyDeviceToHost));
  std::vector<std::pair<int32_t, int32_t>> pr(static_cast<size_t>(found), std::pair<int32_t, int32_t>(0, 0));
  for (size_t k = 0; k < pr.size(); k++) pr[k] = {tmp[2 * k], tmp[2 * k + 1]};
  std::sort(pr.begin(), pr.end());
  const int64_t m = std::min<int64_t>(cap, int64_t(found));
  for (int64_t k = 0; k < m; k++) {
    ij[2 * k]     = pr[size_t(k)].first;
    ij[2 * k + 1] = pr[size_t(k)].second;
  }
  if (int64_t(found) > cap) return fail(MRSB_ERR_CAPACITY, "%llu pairs found, caller buffer holds %lld", found, (long long)cap);
  return MRSB_OK;
}

int mrsb_set_pair_capacity(mrsb_handle h, int64_t max_pairs) {
  GUARD(h);
  if (max_pairs < 1) return fail(MRSB_ERR_INVALID, "max_pairs must be >= 1");
  CU(cudaStreamSynchronize(h->stream));
  int rc = h->pairs.grow(2 * size_t(max_pairs), 2 * size_t(max_pairs), h->stream);
  if (rc) return rc;
  h->grid.pairs    = h->pairs.get();
  h->grid.pair_cap = max_pairs;
  CU(cudaMemsetAsync(h->grid.counters, 0, sizeof(unsigned long long), h->stream));
  return MRSB_OK;
}

int mrsb_get_counters(mrsb_handle h, int64_t* out5) {
  GUARD(h);
  unsigned long long found = 0;
  CU(cudaMemcpyAsync(&found, h->grid.counters, sizeof(found), cudaMemcpyDeviceToHost, h->stream));
  std::vector<uint32_t> fl(size_t(h->ds.n));
  int                   rc = get_flags(h, h->ds.n, nullptr, fl.data());
  if (rc) return rc;
  int64_t crashed = 0;
  for (uint32_t f : fl) crashed += (f & FLAG_CRASHED) ? 1 : 0;
  if (h->lists_on) {
    // table rebuilds happen inside the graph's conditional node: count their kernels from the device-side tally
    NlCtl ctl;
    CU(cudaMemcpy(&ctl, h->grid.ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
    h->n_launches += (int64_t(ctl.n_rebuilds) - h->rebuilds_counted) * h->rebuild_own;
    h->rebuilds_counted = int64_t(ctl.n_rebuilds);
  }
  out5[0] = h->n_steps;
  out5[1] = h->n_passes;
  out5[2] = int64_t(found);
  out5[3] = crashed;
  out5[4] = h->n_launches;
  return MRSB_OK;
}

int mrsb_get_step_info(mrsb_handle h, int32_t* out4) {
  GUARD(h);
  if (!out4) return fail(MRSB_ERR_INVALID, "null output");
  for (int k = 0; k < 4; k++) out4[k] = h->step_info[k];
  return MRSB_OK;
}

int mrsb_get_timeline(mrsb_handle h, uint64_t* out, int64_t max_passes, int64_t* n_passes) {
  GUARD(h);
  CU(cudaStreamSynchronize(h->stream));
  if (n_passes) *n_passes = 0;
  if (!h->grid.tl) return fail(MRSB_ERR_STATE, "no timeline: set MRSB_TIMELINE=1 before mrsb_create");
  NlCtl ctl{};
  CU(cudaMemcpy(&ctl, h->grid.ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
  const int64_t have = std::min<int64_t>(std::min<int64_t>(int64_t(ctl.n_passes), MRSB_TL_TICKS), max_passes);
  if (n_passes) *n_passes = have;
  if (!out || have <= 0) return MRSB_OK;
  // the last `have` passes, oldest first
  std::vector<uint64_t> all(size_t(MRSB_TL_TICKS) * 8);
  CU(cudaMemcpy(all.data(), h->grid.tl, sizeof(uint64_t) * all.size(), cudaMemcpyDeviceToHost));
  for (int64_t k = 0; k < have; k++) {
    const uint64_t pass = ctl.n_passes - uint64_t(have) + uint64_t(k);
    std::memcpy(out + 8 * k, all.data() + (pass % MRSB_TL_TICKS) * 8, sizeof(uint64_t) * 8);
  }
  return MRSB_OK;
}

int mrsb_get_collision_info(mrsb_handle h, double* out8) {
  GUARD(h);
  CU(cudaStreamSynchronize(h->stream));
  NlCtl ctl{};
  if (h->lists_on) CU(cudaMemcpy(&ctl, h->grid.ctl, sizeof(ctl), cudaMemcpyDeviceToHost));
  out8[0] = 1.0 / h->grid.inv_cell;
  out8[1] = h->lists_on ? 1.0 : 0.0;
  out8[2] = h->lists_on ? std::sqrt(h->grid.list_r2) : 0.0;
  out8[3] = h->lists_on ? h->grid.skin : 0.0;
  out8[4] = double(ctl.n_passes);
  out8[5] = double(ctl.n_rebuilds);
  out8[6] = double(ctl.n_crowded);
  out8[7] = double(h->grid.n_buckets);
  return MRSB_OK;
}

// ------------------------------------------------------------------------------------------
// sharded operation
// ------------------------------------------------------------------------------------------
int mrsb_nccl_unique_id(void* out128) {
  int rc = load_nccl();
  if (rc) return rc;
  ncclUniqueId id;
  NC(g_nccl.GetUniqueId(&id));
  std::memcpy(out128, &id, sizeof(id));
  return MRSB_OK;
}

int mrsb_comm_init_nccl(mrsb_handle h, int32_t n_ranks, int32_t rank, const void* unique_id128) {
  GUARD(h);
  int rc = load_nccl();
  if (rc) return rc;
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(MRSB_ERR_INVALID, "bad rank %d of %d", rank, n_ranks);
  ncclUniqueId id;
  std::memcpy(&id, unique_id128, sizeof(id));
  NC(g_nccl.CommInitRank(&h->comm, n_ranks, id, rank));
  h->n_ranks = n_ranks;
  h->rank    = rank;
  // learn every rank's shard with one tiny all-gather
  Mem<int64_t> d_tab;
  rc = d_tab.alloc(2 * size_t(n_ranks));
  if (rc) return rc;
  const int64_t mine[2] = {h->ds.shard_begin, h->ds.n};
  CU(cudaMemcpyAsync(d_tab.get() + 2 * rank, mine, sizeof(mine), cudaMemcpyHostToDevice, h->stream));
  NC(g_nccl.AllGather(d_tab.get() + 2 * rank, d_tab.get(), 2, ncclInt64, h->comm, h->stream));
  std::vector<int64_t> tab(2 * size_t(n_ranks));
  CU(cudaMemcpyAsync(tab.data(), d_tab.get(), sizeof(int64_t) * tab.size(), cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  h->shard_begin_of.assign(size_t(n_ranks), 0);
  h->shard_count_of.assign(size_t(n_ranks), 0);
  h->equal_shards = true;
  int64_t covered = 0;
  for (int r = 0; r < n_ranks; r++) {
    h->shard_begin_of[size_t(r)] = tab[2 * size_t(r)];
    h->shard_count_of[size_t(r)] = tab[2 * size_t(r) + 1];
    covered += tab[2 * size_t(r) + 1];
    if (tab[2 * size_t(r) + 1] != h->ds.n || tab[2 * size_t(r)] != int64_t(r) * h->ds.n) h->equal_shards = false;
  }
  if (covered != h->ds.n_global) return fail(MRSB_ERR_INVALID, "shards cover %lld UAVs, n_global is %lld", (long long)covered, (long long)h->ds.n_global);
  h->ds.n_ranks = n_ranks;
  h->ds.rank    = rank;
  if (n_ranks > 1 && n_ranks <= MRSB_MAX_RANKS && !getenv("MRSB_NO_P2P")) {
    if (setup_p2p(h) != MRSB_OK) {  // no peer access (or IPC refused): the NCCL all-gather stays
      cudaGetLastError();
      h->p2p = false;
    }
  }
  return MRSB_OK;
}

int mrsb_exchange_mode(mrsb_handle h) {
  if (!h) return -1;
  return h->n_ranks <= 1 ? 0 : (h->p2p ? 2 : 1);
}

int mrsb_gather_buffer(mrsb_handle h, void** device_ptr, size_t* bytes) {
  GUARD(h);
  if (device_ptr) *device_ptr = h->ds.gpos;
  if (bytes) *bytes = sizeof(double) * 3 * size_t(h->ds.n_global);
  return MRSB_OK;
}

int mrsb_publish_positions(mrsb_handle h) {
  GUARD(h);
  h->wrote_since_pass  = true;
  h->positions_touched = true;
  h->n_launches += launch_publish_positions(h->ds, h->stream);
  CU(cudaGetLastError());
  return MRSB_OK;
}

int mrsb_get_device_view(mrsb_handle h, mrsb_device_view* out) {
  GUARD(h);
  out->tile        = MRSB_TILE;
  out->state       = h->ds.st;
  out->state_rows  = ST_ROWS;
  out->motor_rpm   = h->ds.rpm;
  out->imu_acc     = h->ds.imu;
  out->ext_force   = h->ds.fext;
  out->flags       = h->ds.flags;
  out->input_mode  = h->ds.mode;
  out->slot_of_uav = h->ds.perm;
  return MRSB_OK;
}

}  // extern "C"
