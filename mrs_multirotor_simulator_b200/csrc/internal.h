// internal.h — device data layout and host bookkeeping of libmrsb (not part of the public ABI).
//
// HBM layout (DESIGN.md §3): tiled structure of arrays ("AoSoA").  Every per-UAV array is cut into
// tiles of MRSB_TILE = 128 consecutive UAVs; inside a tile the ROWS components are stored row after
// row, 128 doubles (1 KiB) each:   element(row, i) = base[((i / 128) * ROWS + row) * 128 + i % 128].
// A 128-thread CTA of the stepping kernel owns exactly one tile: its loads and stores are fully
// coalesced 256-byte warp transactions at COMPILE-TIME offsets from one tile pointer (no per-access
// address arithmetic), and the tile is one contiguous chunk of HBM (DRAM page locality, and one
// bulk copy per array when it is staged through shared memory).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mrsb.h"

#define MRSB_NM MRSB_MAX_MOTORS
#define MRSB_TILE 128

// index of component `row` of UAV `i` in a tiled array with `rows` components
static __host__ __device__ __forceinline__ int64_t tix(int rows, int row, int64_t i) {
  return ((i >> 7) * rows + row) * MRSB_TILE + (i & (MRSB_TILE - 1));
}
// rows of each per-UAV array
#define ST_ROWS 18
#define VPREV_ROWS 3
#define F3_ROWS 3

// per-UAV flag bits
#define FLAG_CRASHED 1u        // UavSystem::crashed_ (US:80)
#define FLAG_TAKEOFF 2u        // live copy of ModelParams::takeoff_patch_enabled (MM:275)
#define FLAG_VPREV 4u          // v_prev array holds a value different from v (after set_state, MM:424-433)
#define FLAG_HAD_INPUT 256u    // a command has arrived at least once (UavSystemRos::time_last_input_ > 0, ROSW:265)
#define FLAG_FF_VEL_HDG_RATE 16u   // std::optional feed-forwards present (US:112-115)
#define FLAG_FF_VEL_HDG 32u
#define FLAG_FF_ACC_HDG_RATE 64u
#define FLAG_FF_ACC_HDG 128u

// rows of the command array (10 payload doubles + cached cos/sin of the heading)
#define CMD_ROWS 12
#define CMD_COS 10
#define CMD_SIN 11
// rows of the feed-forward array
#define FF_VEL_HDG 0       // 3 rows
#define FF_VEL_HDG_RATE 3  // 3 rows
#define FF_ACC_HDG 6       // 3 rows
#define FF_ACC_HDG_RATE 9  // 3 rows + heading_rate
#define FF_ROWS 13
// PID state rows: PID k = 0..2 position xyz, 3..5 velocity xyz, 6..8 attitude xyz, 9..11 rate xyz keeps its last_error in row k
// and its integral in row 12 + k (the integrals of a controller whose ki is zero can then be left out of a launch's traffic)
#define PID_ROWS 24

// One parameter set = one airframe + one set of controller gains, in the form the kernels want.
// Derived on the host (params.cpp) from mrsb_model_params + mrsb_controller_params.
struct DevParams {
  int32_t n_motors;
  int32_t ground_enabled;
  int32_t mixer_desaturation;
  int32_t j_diagonal;
  double  g, mass, inv_mass, inv_kf_n /* 1/(kf*n_motors) */, min_rpm, rpm_range, inv_rpm_range, neg_inv_tau, air_k /* c*pi*l*l */, ground_z,
      takeoff_rpm /* 0.9*hover_rpm, MM:266-267 */;
  double  filt;  // exp(-dt / tau) (MM:244) for the dt of the current launches: evaluated ON THE DEVICE by prep_params_kernel (one
                 // evaluation per parameter set and dt instead of one per UAV and launch; the same bits for every kernel variant)
  double arm_length, prop_radius;  // collision geometry (SIM:342)
  double J[9], Jinv[9];            // row-major
  double alloc[4][MRSB_NM];        // scaled allocation matrix rows: torque xyz, thrust
  double mix[MRSB_NM][4];          // normalised pseudo-inverse (CTL/mixer.hpp:72-101)
  double pos_kp, pos_kd, pos_ki, pos_sat;
  double vel_kp, vel_kd, vel_ki, vel_sat;
  double att_kp, att_kd, att_ki, att_sat_rp, att_sat_yaw;
  double rate_kp[3], rate_kd[3], rate_ki[3];  // already multiplied by J_ii (CTL/rate_controller.hpp:62-64)
};
// The staged stepping kernel takes a DevParams (and a DevState) by value: a field added to either moves the kernel's parameter
// layout, which has been seen to change its register allocation and spills.  What only other kernels need goes beside them:
// the initial take-off flag of every parameter set (mrsb_sim::d_takeoff0), read by the respawn kernels.

// Device pointers of one shard.  Passed to kernels by value.
struct DevState {
  int64_t  n;   // UAVs in this shard
  int64_t  ld;  // n rounded up to a whole number of tiles (allocation size per row)
  double*  st;  // tiled, ST_ROWS rows: x(0-2) v(3-5) R col-major(6-14) omega(15-17)  == InternalState MM:204-214
  double*  vprev;  // [3][ld]  only meaningful where FLAG_VPREV is set
  double*  rpm;    // [MRSB_NM][ld]
  double*  pid;    // [PID_ROWS][ld]
  double*  fext;   // [3][ld] external_force_  (MM:142)
  double*  mext;   // [3][ld] external_moment_ (MM:143)
  double*  imu;    // [3][ld] imu_acceleration_ (MM:139)
  double*  initz;  // [ld] _initial_pos_.z (MM:145; only z is ever read, MM:269-270)
  double*  cmd;    // [CMD_ROWS][ld]
  double*  ff;     // [FF_ROWS][ld]
  uint32_t* flags;  // [ld]
  uint8_t*  mode;   // [ld] INPUT_MODE (US:95)
  const int32_t* pset;  // [n_global] parameter-set index of every UAV of the swarm (local ones at +shard_begin)
  const DevParams* params;
  double* geom;  // [n_global][4] collision geometry {arm_length, prop_radius, mass, 0} of every UAV of the swarm (SIM:342,350); in
                       // pull-exchange runs the slots of remote UAVs are a cache of the owners' values (filled with the halo's positions)
  double*  gpos;  // [n_global][3] packed positions: this shard's slice is written by the step kernel
  int64_t  shard_begin;
  int64_t  n_global;
  // sharded runs with peer access ("pull" exchange): peers read this shard's slice of gpos straight out of this GPU's memory
  // over NVLink.  So that a peer can tell which parts of the slice can matter to it, the step kernel also keeps one bounding
  // box per warp (32 consecutive UAVs): 6 order-preserving uint32 codes of floats rounded outwards, [group][lo xyz, hi xyz].
  uint32_t* gbox;  // [n_groups32][6], nullptr = not tracked
  int64_t   n_groups32;  // (n + 31) / 32
  int32_t  n_ranks, rank;
  uint32_t opts;   // STEP_OPT_* bits
  // Batches with several airframes are BUCKETED at create: the tiled arrays hold the UAVs sorted by airframe, every bucket padded
  // to whole tiles, so that each 128-UAV tile is uniform and the specialised kernels apply.  perm[e] = slot of (external, local)
  // index e; inv[slot] = e, or -1 for a padding slot.  nullptr: identity.  gpos, geom, pset and the neighbour lists stay in
  // external order.
  const int32_t* perm;
  const int32_t* inv;
  // neighbour lists of the collision pass: the stepping kernel atomicMax-es the float bits of the
  // largest squared displacement |x_end - x_start|^2 of this launch here (nullptr = not tracked)
  uint32_t* disp_max;
};

#define STEP_OPT_IMU 1u   // store the fabricated accelerometer rows (MM:280-281); off when nobody reads them (mrsb_set_outputs)
#define STEP_OPT_GPOS 2u  // store the packed positions (collision pass / position download / peers)
#define STEP_OPT_NEED_INPUT 4u  // iterate_without_input == false (ROSW:265): UAVs that never received a command are not stepped

// Sharded runs: where the current position / collision geometry of a global UAV index lives.  n_ranks == 1: everything is in
// this handle's own arrays (single shard, or positions gathered into the local buffer by NCCL or by the caller).
#define MRSB_MAX_RANKS 16
struct PeerView {
  int32_t         n_ranks, rank;
  int64_t         begin[MRSB_MAX_RANKS + 1];  // shard boundaries (global indices)
  const double*   pos[MRSB_MAX_RANKS];        // rank r's packed positions [n_global][3]; only r's own slice is kept current
  const uint32_t* box[MRSB_MAX_RANKS];        // rank r's per-group bounding boxes (DevState::gbox)
  const double*   geom[MRSB_MAX_RANKS];       // rank r's collision geometry [n_global][4]; only r's own slice is kept current
};

// cross-GPU hand-shake of the pull exchange, done by the first kernel of every collision pass (decide_kernel)
struct P2PCtl {
  unsigned long long* const* peer_flags;  // device array [n_ranks]: every rank's flag block (mapped over CUDA IPC)
  unsigned long long*        flags;       // this rank's block: [0, G) pass numbers written by the peers, [G, 3G) their displacement words
  int32_t                    n_ranks, rank;  // n_ranks <= 1: no hand-shake
  int*                       status;      // mapped host word: set to 1 when a peer did not show up in time
  long long                  budget;      // clock64 ticks to wait for a peer
};

// neighbour lists (collide.cu): candidates per UAV kept between table rebuilds
#define MRSB_NL_CAP 8
#define MRSB_TL_TICKS 4096
struct NlCtl {
  uint32_t disp_max_bits;  // written by the stepping kernel (DevState::disp_max points here); 0xFFFFFFFF (a NaN: "unbounded")
                           // makes the pass rebuild: the host raises it before a pass whose bound does not hold (api.cu, begin_pass)
  uint32_t valid;          // lists exist
  uint32_t n_active;       // entries of DevGrid::nl_active (UAVs with something to check on list-only passes)
  uint32_t n_crowded;      // UAVs with more than MRSB_NL_CAP candidates at the last rebuild (they walk the table instead)
  uint32_t rebuild;        // decision of the current pass
  double   D_total;        // sum of the per-launch displacement bounds since the last rebuild
  unsigned long long n_rebuilds, n_passes, epoch /* passes that went through the peer hand-shake */;
  unsigned long long write_all_until;  // host: passes up to this index must write every UAV's force (they were written from outside)
};

// collision pass workspace
struct DevGrid {
  uint32_t  n_buckets;  // power of two >= 2 * n_global
  uint32_t  bits;
  double    inv_cell;   // 1 / cell edge
  double    reach;      // cell / 2: the stencil covers [q - reach, q + reach)
  double    list_r2;    // (sqrt(3) + skin)^2: who goes into a neighbour list
  double    skin;       // lists are valid while 2 * D_total <= skin
  uint32_t* nl_count;   // [nl_ld] candidates of each local UAV; bit 31: its external force may be non-zero (nullptr: no lists)
  int32_t*  nl_items;   // [MRSB_NL_CAP][nl_ld] their global indices, slot-major
  int64_t   nl_ld;
  uint2*    nl_active;  // [n_local] {local index, count word} of the UAVs with a candidate (or the crowded mark), ascending
  int32_t*  act_items;  // [MRSB_NL_CAP][nl_ld] their lists again, slot-major by ENTRY of nl_active (what a list-only pass reads)
  NlCtl*    ctl;
  uint32_t* bucket;     // [n_global] bucket of each UAV, 0xFFFFFFFF = not inserted (remote and outside this shard's box)
  uint32_t* rank;       // [n_global] arrival rank inside its bucket
  uint32_t* count;      // [n_buckets+3] occupancy histogram; [n_buckets], [n_buckets+1] mirror buckets 0 and 1, last entry stays 0
  uint32_t* begin;      // [n_buckets+3] exclusive scan of count; begin[n_buckets] = number of inserted UAVs
  double4*  rec;        // [2*n_global] records {x,y,z, index bits} grouped by bucket (+ the mirror copies of bucket 0)
  unsigned long long* aabb;  // [6] order-preserving encoding of min xyz / max xyz of this shard's positions
  unsigned long long* scan_state;  // [1 + tiles] ticket counter + per-tile status words of the single-pass prefix sum
  int32_t   scan_tiles;
  // pull exchange: remote UAVs that can reach this shard's box, fetched from their owners at a rebuild
  double4*  halo_rec;   // [halo_cap] {x, y, z, global index}
  uint32_t* halo_bucket, *halo_rank;  // [halo_cap]
  uint32_t* halo_n;     // device counter; halo_n[1] = halo_work_n
  uint32_t* halo_work;  // [groups of all peers] work list of a rebuild: (rank << 26 | group) of the remote 32-UAV groups that can reach this shard
  uint32_t* halo_work_n;
  int64_t   halo_cap;
  // diagnostics (MRSB_TIMELINE=1 at create): %globaltimer stamps of the pass' kernels, [MRSB_TL_TICKS][8] indexed by pass number:
  // 0 decide start, 1 hand-shake sent, 2 hand-shake complete, 3 halo refresh start, 4 list check start, 5 rebuild flag, 6 table build start, 7 list build start
  unsigned long long* tl;
  int32_t*  pairs;      // [pair_cap][2]
  int64_t   pair_cap;
  unsigned long long* counters;  // [0] pairs found by the last pass
};

// kernel launchers (step_kernel.cu / collide.cu / io_kernels.cu); all return the number of launches made
// uniform_params: host copy of THE parameter set when every local UAV uses the same one, else nullptr
// sweep: the launch's own device word, zero at first use, whose parity sets the direction of the staged kernel's sweep; nullptr:
// always forward (the staged kernel also sweeps forward when its launch streams less than L2 holds)
// info[4] (may be nullptr): [0] variant launched — 1 direct (one CTA per tile), 2 staged (persistent CTAs + TMA); [1] grid;
// [2] NM_T and [3] MODE_T of the instantiation
int launch_step(const DevState& s, const DevParams* uniform_params, uint32_t* sweep, double dt, int k_substeps, int uniform_mode, int uniform_nm, bool any_moment,
                cudaStream_t stream, int* info);
// DevParams::filt = exp(dt * neg_inv_tau) for every parameter set of the table
int launch_prep_params(DevParams* params, int n_sets, double dt, cudaStream_t stream);
// The full pass of every tick (handles without neighbour lists): [hand-shake,] table, collide_kernel
int launch_collide(const DevState& s, const DevGrid& g, const PeerView& pv, const P2PCtl& p2p, int crash_mode, double rebounce, cudaStream_t stream);
// the pass with neighbour lists: decide (always; includes the peer hand-shake) | rebuild (body of the graph's conditional node) | check (always)
int launch_collide_decide(const DevGrid& g, const P2PCtl& p2p, int always, cudaGraphConditionalHandle handle, int has_handle, cudaStream_t stream);
int launch_collide_rebuild(const DevState& s, const DevGrid& g, const PeerView& pv, cudaStream_t stream);
int launch_collide_check(const DevState& s, const DevGrid& g, const PeerView& pv, int crash_mode, double rebounce, int beside_rebuild, cudaStream_t stream);
int scan_tiles_for(int64_t n_items);
// Neighbour observations (mrsb_pack_neighbours_device) of a single-shard handle: the table over the workspace `t` (only its table
// fields are read: n_buckets, inv_cell, reach, bucket, rank, count, begin, rec, scan_state, scan_tiles), pos / vel its packed rows
// [n][3]; r2 = radius * radius; outputs as in include/mrsb.h (any may be nullptr)
int launch_neighbours(const DevState& s, const DevGrid& t, double* pos, double* vel, double r2, int k, int32_t* idx, double* rows, int stride,
                      int32_t* count, cudaStream_t stream);
int launch_publish_positions(const DevState& s, cudaStream_t stream);

int launch_scatter_input(const DevState& s, int mode, int64_t n, const int32_t* idx_dev, const double* payload_dev, int stride, cudaStream_t stream);
// row k (k < n <= INT32_MAX) sets UAV idx_dev[k] to mode modes_dev[k] with payload row k; of several rows for one UAV the last wins.
// last_dev: one int32 per slot (s.ld), -1 before and after the call.
int launch_input_rows(const DevState& s, int64_t n, const int32_t* idx_dev, const int32_t* modes_dev, const double* payload_dev, int stride,
                      int32_t* last_dev, cudaStream_t stream);
// payload[k][0..rows) <-> rows [row0, row0+rows) of a tiled array with `rows_total` components
int launch_scatter_rows(double* dst, int rows_total, int row0, int rows, int64_t n, const int32_t* idx_dev, const double* payload_dev, int stride,
                        const int32_t* perm, cudaStream_t stream);
int launch_gather_rows(const double* src, int rows_total, int row0, int rows, int64_t n, const int32_t* idx_dev, double* out_dev, int stride,
                       const int32_t* perm, cudaStream_t stream);
int launch_flag_update(const DevState& s, int64_t n, const int32_t* idx_dev, uint32_t and_mask, uint32_t or_mask, cudaStream_t stream);
int launch_gather_u32(const uint32_t* src, int64_t n, const int32_t* idx_dev, uint32_t* out_dev, const int32_t* perm, cudaStream_t stream);
int launch_gather_u8(const uint8_t* src, int64_t n, const int32_t* idx_dev, int32_t* out_dev, const int32_t* perm, cudaStream_t stream);
int launch_set_mode(const DevState& s, int64_t n, const int32_t* idx_dev, int mode, cudaStream_t stream);
int launch_set_state_pos(const DevState& s, int64_t n, const int32_t* idx_dev, const double* xyz_dev, const double* hdg_dev, cudaStream_t stream);
// UavSystem(params, pos, heading) again for the addressed UAVs (payload rows k) / for every UAV e with mask[e] != 0 (payload rows
// e; raises the displacement word when it respawned anybody).  takeoff0[set]: initial take-off flag of each parameter set.
int launch_respawn(const DevState& s, const uint8_t* takeoff0, int64_t n, const int32_t* idx_dev, const double* xyz_dev, const double* hdg_dev,
                   cudaStream_t stream);
int launch_respawn_masked(const DevState& s, const uint8_t* takeoff0, const uint8_t* mask_dev, const double* xyz_dev, const double* hdg_dev,
                          cudaStream_t stream);
// Snapshots (mrsb_snapshot_*): rows [SNAP_ROWS][s.n] doubles, flags [s.n], mode [s.n], all in external order.  save: every UAV.
// restore: UAV idx[k] (nullptr: k) takes record src[k] (nullptr: its own), k < n.  restore_masked: UAV e takes record src[e]
// when 0 <= src[e] < s.n (src == nullptr: its own), else is left alone; raises the displacement word when it restored anybody.
#define SNAP_ROWS 88
int launch_snapshot_save(const DevState& s, double* rows, uint32_t* flags, uint8_t* mode, cudaStream_t stream);
int launch_snapshot_restore(const DevState& s, const double* rows, const uint32_t* flags, const uint8_t* mode, int64_t n, const int32_t* idx_dev,
                            const int32_t* src_dev, cudaStream_t stream);
int launch_snapshot_restore_masked(const DevState& s, const double* rows, const uint32_t* flags, const uint8_t* mode, const int32_t* src_dev,
                                   cudaStream_t stream);
int launch_stash_vprev(const DevState& s, int64_t n, const int32_t* idx_dev, cudaStream_t stream);
int launch_gather_vprev(const DevState& s, int64_t n, const int32_t* idx_dev, double* out_dev, cudaStream_t stream);
// zero the state (last error and integral) of PIDs [pid0, pid0 + n_pids)
int launch_reset_pid(const DevState& s, int64_t n, const int32_t* idx_dev, int pid0, int n_pids, cudaStream_t stream);
int launch_timeout_input(const DevState& s, int64_t n, const int32_t* idx_dev, cudaStream_t stream);
int launch_gather_xyz(const double* xyz_dev, int64_t n, const int32_t* idx_dev, double* out_dev, cudaStream_t stream);
int launch_tracker_cmd(const DevState& s, int64_t n, const int32_t* idx_dev, const double* rows_dev, cudaStream_t stream);
int launch_observe(const DevState& s, int what, int64_t n, const int32_t* idx_dev, double* out_dev, int stride, cudaStream_t stream);
int launch_set_pset(int32_t* pset_dev, int64_t n, const int32_t* idx_dev, int64_t offset, const int32_t* values_dev, cudaStream_t stream);
// geom[j] = {arm, prop radius, mass, 0} of params[pset[j]] for j = offset + idx[k] (idx == nullptr: j = offset + k), k < n
int launch_set_geom(double* geom_dev, int64_t n, const int32_t* idx_dev, int64_t offset, const int32_t* pset_dev, const DevParams* params, cudaStream_t stream);
