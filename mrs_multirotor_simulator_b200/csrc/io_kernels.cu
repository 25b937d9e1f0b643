// io_kernels.cu — row-per-UAV (caller side) <-> structure-of-arrays (device side) movers behind the
// setInput / getState / applyForce ... entry points of the C ABI.  One thread per addressed UAV;
// idx == nullptr means "UAV k" (identity).
#include "internal.h"

namespace {

#define DEV __device__ __forceinline__
// k-th addressed UAV: its (external) local index ...
DEV int64_t ext(const int32_t* idx, int64_t k) { return idx ? int64_t(idx[k]) : k; }
// ... and the slot of the tiled arrays it lives in: the identity unless the batch was bucketed by airframe at create
// (DevState::perm, api.cu) so that every 128-UAV tile holds one airframe
DEV int64_t at(const int32_t* perm, const int32_t* idx, int64_t k) {
  const int64_t e = ext(idx, k);
  return perm ? int64_t(perm[e]) : e;
}

inline unsigned nblk(int64_t n, int t = 256) { return unsigned((n + t - 1) / t); }

// UavSystem::setInput overloads (US:175-248) for the UAV in slot i: store the command row p[0 .. stride), switch the mode.  cos/sin
// of the commanded heading (used by CTL/acceleration_controller.hpp:50) are cached once per command instead of being re-evaluated
// every step.
DEV void apply_input(const DevState& s, int mode, int64_t i, const double* __restrict__ p, int stride) {
  const int rows = mode == MRSB_ACTUATOR_CMD ? MRSB_NM : (mode == MRSB_ATTITUDE_CMD ? 10 : (mode == MRSB_TILT_HDG_RATE_CMD ? 5 : 4));
  for (int r = 0; r < rows; r++) s.cmd[tix(CMD_ROWS, r, i)] = r < stride ? p[r] : 0.0;
  if (mode == MRSB_POSITION_CMD || mode == MRSB_VELOCITY_HDG_CMD || mode == MRSB_ACCELERATION_HDG_CMD) {
    double sn, cs;
    sincos(p[3], &sn, &cs);
    s.cmd[tix(CMD_ROWS, CMD_COS, i)] = cs;
    s.cmd[tix(CMD_ROWS, CMD_SIN, i)] = sn;
  }
  s.mode[i] = uint8_t(mode);
  if (!(s.flags[i] & FLAG_HAD_INPUT)) s.flags[i] |= FLAG_HAD_INPUT;  // time_last_input_ > 0 from now on (ROSW:265)
}

__global__ void scatter_input_kernel(DevState s, int mode, int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ payload, int stride) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t e = ext(idx, k);
  if (e < 0 || e >= s.n) return;
  const int64_t i = s.perm ? int64_t(s.perm[e]) : e;
  apply_input(s, mode, i, payload + k * stride, stride);
}

// Mixed-mode command rows (mrsb_set_input_rows_async): row k sets UAV idx[k] to mode modes[k], and of several rows for one UAV the
// last one wins — without sorting.  last[slot] is a persistent word that holds -1 between calls.  The claim kernel leaves in it the
// highest row number addressed to the slot; in the apply kernel that row alone applies itself and puts the -1 back.  A losing row
// reads the winner's number or, once the winner is done, -1: either way not its own, so it skips.
__global__ void input_rows_claim_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx, int32_t* __restrict__ last) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  atomicMax(&last[at(s.perm, idx, k)], int32_t(k));
}

__global__ void input_rows_apply_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx, const int32_t* __restrict__ modes,
                                        const double* __restrict__ payload, int stride, int32_t* last) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i = at(s.perm, idx, k);
  if (last[i] != int32_t(k)) return;
  apply_input(s, modes[k], i, payload + k * stride, stride);
  last[i] = -1;
}

__global__ void set_mode_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx, int mode) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t e = ext(idx, k);
  if (e < 0 || e >= s.n) return;
  const int64_t i = s.perm ? int64_t(s.perm[e]) : e;
  s.mode[i] = uint8_t(mode);
}

// payload[k][0 .. rows) -> rows [row0, row0+rows) of UAV i
__global__ void scatter_rows_kernel(double* __restrict__ dst, int rows_total, int row0, int rows, int64_t n, const int32_t* __restrict__ idx,
                                    const double* __restrict__ payload, int stride, const int32_t* __restrict__ perm) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i = at(perm, idx, k);
  for (int r = 0; r < rows; r++) dst[tix(rows_total, row0 + r, i)] = payload[k * stride + r];
}

__global__ void gather_rows_kernel(const double* __restrict__ src, int rows_total, int row0, int rows, int64_t n, const int32_t* __restrict__ idx,
                                   double* __restrict__ out, int stride, const int32_t* __restrict__ perm) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i = at(perm, idx, k);
  for (int r = 0; r < rows; r++) out[k * stride + r] = src[tix(rows_total, row0 + r, i)];
}

__global__ void flag_update_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx, uint32_t and_mask, uint32_t or_mask) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i = at(s.perm, idx, k);
  s.flags[i]      = (s.flags[i] & and_mask) | or_mask;
}

__global__ void gather_u32_kernel(const uint32_t* __restrict__ src, int64_t n, const int32_t* __restrict__ idx, uint32_t* __restrict__ out,
                                  const int32_t* __restrict__ perm) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  out[k] = src[at(perm, idx, k)];
}

__global__ void gather_u8_kernel(const uint8_t* __restrict__ src, int64_t n, const int32_t* __restrict__ idx, int32_t* __restrict__ out,
                                 const int32_t* __restrict__ perm) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  out[k] = int32_t(src[at(perm, idx, k)]);
}

// MultirotorModel::setStatePos (MM:439-446) of the UAV in slot i, external index e: x, _initial_pos_, R = AngleAxis(-heading, z)
DEV void write_pose(const DevState& s, int64_t i, int64_t e, double px, double py, double pz, double neg_hdg) {
  double sn, cs;
  sincos(neg_hdg, &sn, &cs);
  s.st[tix(ST_ROWS, 0, i)] = px;
  s.st[tix(ST_ROWS, 1, i)] = py;
  s.st[tix(ST_ROWS, 2, i)] = pz;
  s.initz[i]       = pz;
  // column-major R = [[c,-s,0],[s,c,0],[0,0,(1-c)+c]] for angle -heading (Eigen AngleAxis::toRotationMatrix)
  s.st[tix(ST_ROWS, 6, i)]  = cs;
  s.st[tix(ST_ROWS, 7, i)]  = sn;
  s.st[tix(ST_ROWS, 8, i)]  = 0.0;
  s.st[tix(ST_ROWS, 9, i)]  = -sn;
  s.st[tix(ST_ROWS, 10, i)] = cs;
  s.st[tix(ST_ROWS, 11, i)] = 0.0;
  s.st[tix(ST_ROWS, 12, i)] = 0.0;
  s.st[tix(ST_ROWS, 13, i)] = 0.0;
  s.st[tix(ST_ROWS, 14, i)] = (1.0 - cs) + cs;
  double* gp        = s.gpos + 3 * (s.shard_begin + e);
  gp[0]             = px;
  gp[1]             = py;
  gp[2]             = pz;
}

__global__ void set_state_pos_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ xyz,
                                     const double* __restrict__ hdg) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t e = ext(idx, k);
  write_pose(s, s.perm ? int64_t(s.perm[e]) : e, e, xyz ? xyz[3 * k] : 0.0, xyz ? xyz[3 * k + 1] : 0.0, xyz ? xyz[3 * k + 2] : 0.0,
             hdg ? -hdg[k] : -0.0);
}

// UavSystem(params, pos, heading) (US:144-153 -> MM:183-198 + MM:439-446) for the UAV in slot i, external index e, keeping its
// parameter set (airframe, edits, controller gains): everything a fresh handle holds after mrsb_create.  v_prev is not written:
// with FLAG_VPREV clear it reads as v.
DEV void respawn_one(const DevState& s, const uint8_t* takeoff0, int64_t i, int64_t e, double px, double py, double pz, double hdg) {
  write_pose(s, i, e, px, py, pz, -hdg);
  for (int r = 3; r < 6; r++) s.st[tix(ST_ROWS, r, i)] = 0.0;  // v
  for (int r = 15; r < ST_ROWS; r++) s.st[tix(ST_ROWS, r, i)] = 0.0;  // omega
  for (int r = 0; r < MRSB_NM; r++) s.rpm[tix(MRSB_NM, r, i)] = 0.0;
  for (int r = 0; r < PID_ROWS; r++) s.pid[tix(PID_ROWS, r, i)] = 0.0;  // CTL/*::setParams reset every PID
  for (int r = 0; r < CMD_ROWS; r++) s.cmd[tix(CMD_ROWS, r, i)] = 0.0;
  for (int r = 0; r < FF_ROWS; r++) s.ff[tix(FF_ROWS, r, i)] = 0.0;
  for (int r = 0; r < F3_ROWS; r++) {
    s.fext[tix(F3_ROWS, r, i)] = 0.0;
    s.mext[tix(F3_ROWS, r, i)] = 0.0;
    s.imu[tix(F3_ROWS, r, i)]  = 0.0;
  }
  s.mode[i]  = uint8_t(MRSB_INPUT_UNKNOWN);
  // crashed, v_prev, feed-forwards and "had a command" cleared; the take-off patch as the parameter set carries it (MM:87)
  s.flags[i] = takeoff0[s.pset[s.shard_begin + e]] ? FLAG_TAKEOFF : 0u;
}

__global__ void respawn_kernel(DevState s, const uint8_t* __restrict__ takeoff0, int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ xyz, const double* __restrict__ hdg) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t e = ext(idx, k);
  respawn_one(s, takeoff0, s.perm ? int64_t(s.perm[e]) : e, e, xyz[3 * k], xyz[3 * k + 1], xyz[3 * k + 2], hdg[k]);
}

// One thread per SLOT (tile order), so that a warp's stores to a row of the tiled arrays are coalesced when many UAVs respawn.
// A respawned UAV moved behind the stepping kernel's displacement bound: the displacement word is raised to "unbounded" (read as
// NaN by decide_kernel: the next pass rebuilds, and in pull-exchange runs the word travels to every peer) — one atomic per warp
// that respawned anybody, none otherwise.
__global__ void respawn_masked_kernel(DevState s, const uint8_t* __restrict__ takeoff0, const uint8_t* __restrict__ mask, const double* __restrict__ xyz, const double* __restrict__ hdg) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  int64_t       e = -1;
  if (i < s.ld) e = s.inv ? int64_t(s.inv[i]) : (i < s.n ? i : -1);
  const bool hit = e >= 0 && mask[e] != 0;
  if (hit) respawn_one(s, takeoff0, i, e, xyz[3 * e], xyz[3 * e + 1], xyz[3 * e + 2], hdg[e]);
  if (s.disp_max && __ballot_sync(0xffffffffu, hit) && (threadIdx.x & 31) == 0) atomicMax(s.disp_max, 0xFFFFFFFFu);
}

// Snapshot record of the UAV in slot i (mrsb_snapshot_*): f(row, element) for every double row in record order — st 0-17, rpm
// 18-25, pid 26-49, cmd 50-61, ff 62-74, fext 75-77, mext 78-80, imu 81-83, vprev 84-86, initz 87 (SNAP_ROWS).
template <class F>
DEV void for_each_record_row(const DevState& s, int64_t i, F f) {
  int r = 0;
#pragma unroll
  for (int k = 0; k < ST_ROWS; k++) f(r++, s.st[tix(ST_ROWS, k, i)]);
#pragma unroll
  for (int k = 0; k < MRSB_NM; k++) f(r++, s.rpm[tix(MRSB_NM, k, i)]);
#pragma unroll
  for (int k = 0; k < PID_ROWS; k++) f(r++, s.pid[tix(PID_ROWS, k, i)]);
#pragma unroll
  for (int k = 0; k < CMD_ROWS; k++) f(r++, s.cmd[tix(CMD_ROWS, k, i)]);
#pragma unroll
  for (int k = 0; k < FF_ROWS; k++) f(r++, s.ff[tix(FF_ROWS, k, i)]);
#pragma unroll
  for (int k = 0; k < F3_ROWS; k++) f(r++, s.fext[tix(F3_ROWS, k, i)]);
#pragma unroll
  for (int k = 0; k < F3_ROWS; k++) f(r++, s.mext[tix(F3_ROWS, k, i)]);
#pragma unroll
  for (int k = 0; k < F3_ROWS; k++) f(r++, s.imu[tix(F3_ROWS, k, i)]);
#pragma unroll
  for (int k = 0; k < VPREV_ROWS; k++) f(r++, s.vprev[tix(VPREV_ROWS, k, i)]);
  f(r, s.initz[i]);
}
static_assert(ST_ROWS + MRSB_NM + PID_ROWS + CMD_ROWS + FF_ROWS + 3 * F3_ROWS + VPREV_ROWS + 1 == SNAP_ROWS, "snapshot record rows");

// One thread per slot (tile order): the reads of the tiled rows are coalesced, the writes go to the external index, which is
// contiguous within a bucket.  Padding slots are skipped.
__global__ void snapshot_save_kernel(DevState s, double* __restrict__ rows, uint32_t* __restrict__ flags, uint8_t* __restrict__ mode) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= s.ld) return;
  const int64_t e = s.inv ? int64_t(s.inv[i]) : (i < s.n ? i : -1);
  if (e < 0) return;
  for_each_record_row(s, i, [&](int r, const double& v) { rows[r * s.n + e] = v; });
  flags[e] = s.flags[i];
  mode[e]  = s.mode[i];
}

// the UAV in slot i, external index e, takes saved record j: every row of the record, its flags and input mode, and its packed
// position (what the collision pass, position downloads and publish_positions read), as write_pose does for a respawn
DEV void restore_one(const DevState& s, const double* __restrict__ rows, const uint32_t* __restrict__ flags, const uint8_t* __restrict__ mode,
                     int64_t i, int64_t e, int64_t j) {
  for_each_record_row(s, i, [&](int r, double& v) { v = rows[r * s.n + j]; });
  s.flags[i] = flags[j];
  s.mode[i]  = mode[j];
  double* gp = s.gpos + 3 * (s.shard_begin + e);
  gp[0]      = rows[0 * s.n + j];
  gp[1]      = rows[1 * s.n + j];
  gp[2]      = rows[2 * s.n + j];
}

// host form: pair k = (UAV idx[k], record src[k]); idx == nullptr: UAV k, src == nullptr: its own record
__global__ void snapshot_restore_kernel(DevState s, const double* __restrict__ rows, const uint32_t* __restrict__ flags, const uint8_t* __restrict__ mode,
                                        int64_t n, const int32_t* __restrict__ idx, const int32_t* __restrict__ src) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t e = ext(idx, k);
  restore_one(s, rows, flags, mode, s.perm ? int64_t(s.perm[e]) : e, e, src ? int64_t(src[k]) : e);
}

// device form, one thread per slot: UAV e takes record src[e] when 0 <= src[e] < n (src == nullptr: its own), else is left alone.
// A restored UAV moved behind the stepping kernel's displacement bound: as in respawn_masked_kernel, one atomic per warp that
// restored anybody raises the displacement word to "unbounded".
__global__ void snapshot_restore_masked_kernel(DevState s, const double* __restrict__ rows, const uint32_t* __restrict__ flags,
                                               const uint8_t* __restrict__ mode, const int32_t* __restrict__ src) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  int64_t       e = -1, j = -1;
  if (i < s.ld) e = s.inv ? int64_t(s.inv[i]) : (i < s.n ? i : -1);
  if (e >= 0) j = src ? int64_t(src[e]) : e;
  const bool hit = j >= 0 && j < s.n;
  if (hit) restore_one(s, rows, flags, mode, i, e, j);
  if (s.disp_max && __ballot_sync(0xffffffffu, hit) && (threadIdx.x & 31) == 0) atomicMax(s.disp_max, 0xFFFFFFFFu);
}

// before set_state overwrites v: remember the old v as v_prev (MM:424-433 leaves v_prev alone)
__global__ void stash_vprev_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i = at(s.perm, idx, k);
  if (s.flags[i] & FLAG_VPREV) return;
  for (int r = 0; r < 3; r++) s.vprev[tix(VPREV_ROWS, r, i)] = s.st[tix(ST_ROWS, 3 + r, i)];
  s.flags[i] |= FLAG_VPREV;
}

__global__ void gather_vprev_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx, double* __restrict__ out) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i  = at(s.perm, idx, k);
  const bool    ov = s.flags[i] & FLAG_VPREV;
  for (int r = 0; r < 3; r++) out[3 * k + r] = ov ? s.vprev[tix(VPREV_ROWS, r, i)] : s.st[tix(ST_ROWS, 3 + r, i)];
}

__global__ void reset_pid_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx, int pid0, int n_pids) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i = at(s.perm, idx, k);
  for (int r = pid0; r < pid0 + n_pids; r++) {
    s.pid[tix(PID_ROWS, r, i)]      = 0.0;  // last error
    s.pid[tix(PID_ROWS, 12 + r, i)] = 0.0;  // integral
  }
}

__global__ void set_pset_kernel(int32_t* __restrict__ pset, int64_t n, const int32_t* __restrict__ idx, int64_t offset,
                                const int32_t* __restrict__ values) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  pset[offset + ext(idx, k)] = values[k];
}

// UavSystemRos::callbackTrackerCmd (ROSW:987-1022): one tracker command row -> the four sticky feed-forwards.
// row[11] = velocity xyz | acceleration xyz | heading_rate | use_velocity_horizontal | use_velocity_vertical | use_heading_rate | use_acceleration
__global__ void tracker_cmd_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx, const double* __restrict__ rows) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i  = at(s.perm, idx, k);
  const double* r  = rows + MRSB_TRACKER_CMD_STRIDE * k;
  const bool    uh = r[7] != 0.0, uv = r[8] != 0.0, ur = r[9] != 0.0, ua = r[10] != 0.0;
  const double  v[3] = {uh ? r[0] : 0.0, uh ? r[1] : 0.0, uv ? r[2] : 0.0};
  const double  a[3] = {ua ? r[3] : 0.0, ua ? r[4] : 0.0, ua ? r[5] : 0.0};
  for (int c = 0; c < 3; c++) {
    s.ff[tix(FF_ROWS, FF_VEL_HDG + c, i)]      = v[c];
    s.ff[tix(FF_ROWS, FF_VEL_HDG_RATE + c, i)] = v[c];
    s.ff[tix(FF_ROWS, FF_ACC_HDG + c, i)]      = a[c];
    s.ff[tix(FF_ROWS, FF_ACC_HDG_RATE + c, i)] = a[c];
  }
  s.ff[tix(FF_ROWS, FF_ACC_HDG_RATE + 3, i)] = ur ? r[6] : 0.0;
  s.flags[i] |= FLAG_FF_VEL_HDG | FLAG_FF_VEL_HDG_RATE | FLAG_FF_ACC_HDG | FLAG_FF_ACC_HDG_RATE;
}

// packed positions of a subset: out[k] = xyz[idx[k]] (both packed [.][3])
__global__ void gather_xyz_kernel(const double* __restrict__ xyz, int64_t n, const int32_t* __restrict__ idx, double* __restrict__ out) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const double* p = xyz + 3 * int64_t(idx[k]);
  out[3 * k] = p[0], out[3 * k + 1] = p[1], out[3 * k + 2] = p[2];
}

// collision geometry of the addressed UAVs from their parameter set
__global__ void set_geom_kernel(double* __restrict__ geom, int64_t n, const int32_t* __restrict__ idx, int64_t offset, const int32_t* __restrict__ pset,
                                const DevParams* __restrict__ params) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t    j = offset + ext(idx, k);
  const DevParams& P = params[pset[j]];
  geom[4 * j + 0]    = P.arm_length;
  geom[4 * j + 1]    = P.prop_radius;
  geom[4 * j + 2]    = P.mass;
  geom[4 * j + 3]    = 0.0;
}

// UavSystemRos::timeoutInput (ROSW:474-647): the active command becomes its "hover" version
__global__ void timeout_input_kernel(DevState s, int64_t n, const int32_t* __restrict__ idx) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i    = at(s.perm, idx, k);
  const int     mode = s.mode[i];
  s.flags[i] &= ~FLAG_HAD_INPUT;  // time_last_input_ = 0 (ROSW:256-259): with iterate_without_input off the UAV stops until the next command
  auto          C    = [&](int row) -> double& { return s.cmd[tix(CMD_ROWS, row, i)]; };
  auto          S    = [&](int row) { return s.st[tix(ST_ROWS, row, i)]; };
  const double  hdg  = atan2(S(7), S(6));  // AttitudeConverter(R).getHeading(): atan2(R10, R00)
  double        sh, ch;
  sincos(hdg, &sh, &ch);
  switch (mode) {
    case MRSB_POSITION_CMD:
      C(0) = S(0), C(1) = S(1), C(2) = S(2), C(3) = hdg, C(CMD_COS) = ch, C(CMD_SIN) = sh;
      break;
    case MRSB_VELOCITY_HDG_CMD:
    case MRSB_ACCELERATION_HDG_CMD:
      C(0) = 0.0, C(1) = 0.0, C(2) = 0.0, C(3) = hdg, C(CMD_COS) = ch, C(CMD_SIN) = sh;
      break;
    case MRSB_VELOCITY_HDG_RATE_CMD:
    case MRSB_ACCELERATION_HDG_RATE_CMD:
    case MRSB_ATTITUDE_RATE_CMD:
    case MRSB_CONTROL_GROUP_CMD:
      C(0) = 0.0, C(1) = 0.0, C(2) = 0.0, C(3) = 0.0;
      break;
    case MRSB_ATTITUDE_CMD:  // AttitudeConverter(0, 0, heading) -> Rz(heading), column-major; throttle 0
      C(0) = ch, C(1) = sh, C(2) = 0.0, C(3) = -sh, C(4) = ch, C(5) = 0.0, C(6) = 0.0, C(7) = 0.0, C(8) = 1.0, C(9) = 0.0;
      break;
    case MRSB_TILT_HDG_RATE_CMD:
      C(0) = 0.0, C(1) = 0.0, C(2) = 1.0, C(3) = 0.0, C(4) = 0.0;
      break;
    case MRSB_ACTUATOR_CMD:
      for (int m = 0; m < MRSB_NM; m++) C(m) = 0.0;
      break;
    default:
      break;
  }
}

// Eigen::Quaterniond(Matrix3d) as used by mrs_lib::AttitudeConverter(R); q = x y z w
DEV void quaternion_of(const double* m /* column-major */, double* q) {
  auto   M = [&](int r, int c) { return m[3 * c + r]; };
  double t = M(0, 0) + (M(1, 1) + M(2, 2));
  if (t > 0.0) {
    t    = sqrt(t + 1.0);
    q[3] = 0.5 * t;
    t    = 0.5 / t;
    q[0] = (M(2, 1) - M(1, 2)) * t;
    q[1] = (M(0, 2) - M(2, 0)) * t;
    q[2] = (M(1, 0) - M(0, 1)) * t;
  } else {
    int i = 0;
    if (M(1, 1) > M(0, 0)) i = 1;
    if (M(2, 2) > M(i, i)) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t    = sqrt(M(i, i) - M(j, j) - M(k, k) + 1.0);
    q[i] = 0.5 * t;
    t    = 0.5 / t;
    q[3] = (M(k, j) - M(j, k)) * t;
    q[j] = (M(j, i) + M(i, j)) * t;
    q[k] = (M(k, i) + M(i, k)) * t;
  }
}

// what = 0: publishOdometry (ROSW:340-368) rows [13]; 1: publishIMU (ROSW:374-395) rows [10];
// 2: publishRangefinder (ROSW:401-420) rows [1]; 3: all of them packed for device-resident callers, rows [17] =
// odometry 13 | IMU linear acceleration 3 | range 1
__global__ void observe_kernel(DevState s, int what, int64_t n, const int32_t* __restrict__ idx, double* __restrict__ out, int stride) {
  const int64_t k = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t e = ext(idx, k);
  const int64_t i = s.perm ? int64_t(s.perm[e]) : e;
  double        x[3], v[3], R[9], w[3], q[4];
  for (int r = 0; r < 3; r++) {
    x[r] = s.st[tix(ST_ROWS, r, i)];
    v[r] = s.st[tix(ST_ROWS, 3 + r, i)];
    w[r] = s.st[tix(ST_ROWS, 15 + r, i)];
  }
  for (int r = 0; r < 9; r++) R[r] = s.st[tix(ST_ROWS, 6 + r, i)];
  double* o = out + k * stride;
  if (what == 0 || what == 1 || what == 3) quaternion_of(R, q);
  double range = 0.0;
  if (what == 2 || what == 3) {
    const double bz   = R[8];
    const double tilt = acos((-R[6]) * 0.0 + ((-R[7]) * 0.0 + (-bz) * -1.0));
    range             = bz > 0.0 ? (x[2] - s.params[s.pset[s.shard_begin + e]].ground_z) / cos(tilt) + 0.01 : 1.7976931348623157e308;
    if (range > 40.0) range = 41.0;
  }
  if (what == 0 || what == 3) {
    for (int r = 0; r < 3; r++) o[r] = x[r];
    for (int r = 0; r < 4; r++) o[3 + r] = q[r];
    for (int r = 0; r < 3; r++) {
      o[7 + r]  = R[3 * r] * v[0] + (R[3 * r + 1] * v[1] + R[3 * r + 2] * v[2]);  // R^T v
      o[10 + r] = w[r];
    }
    if (what == 3) {
      for (int r = 0; r < 3; r++) o[13 + r] = s.imu[tix(F3_ROWS, r, i)];
      o[16] = range;
    }
  } else if (what == 1) {
    for (int r = 0; r < 3; r++) {
      o[r]     = w[r];
      o[3 + r] = s.imu[tix(F3_ROWS, r, i)];
    }
    for (int r = 0; r < 4; r++) o[6 + r] = q[r];
  } else {
    o[0] = range;
  }
}

}  // namespace

int launch_timeout_input(const DevState& s, int64_t n, const int32_t* idx, cudaStream_t st) {
  if (n <= 0) return 0;
  timeout_input_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx);
  return 1;
}
int launch_observe(const DevState& s, int what, int64_t n, const int32_t* idx, double* out, int stride, cudaStream_t st) {
  if (n <= 0) return 0;
  observe_kernel<<<nblk(n), 256, 0, st>>>(s, what, n, idx, out, stride);
  return 1;
}

int launch_scatter_input(const DevState& s, int mode, int64_t n, const int32_t* idx, const double* payload, int stride, cudaStream_t st) {
  if (n <= 0) return 0;
  scatter_input_kernel<<<nblk(n), 256, 0, st>>>(s, mode, n, idx, payload, stride);
  return 1;
}
int launch_input_rows(const DevState& s, int64_t n, const int32_t* idx, const int32_t* modes, const double* payload, int stride, int32_t* last,
                      cudaStream_t st) {
  if (n <= 0) return 0;
  input_rows_claim_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx, last);
  input_rows_apply_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx, modes, payload, stride, last);
  return 2;
}
int launch_set_mode(const DevState& s, int64_t n, const int32_t* idx, int mode, cudaStream_t st) {
  if (n <= 0) return 0;
  set_mode_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx, mode);
  return 1;
}
int launch_scatter_rows(double* dst, int rows_total, int row0, int rows, int64_t n, const int32_t* idx, const double* payload, int stride,
                        const int32_t* perm, cudaStream_t st) {
  if (n <= 0) return 0;
  scatter_rows_kernel<<<nblk(n), 256, 0, st>>>(dst, rows_total, row0, rows, n, idx, payload, stride, perm);
  return 1;
}
int launch_gather_rows(const double* src, int rows_total, int row0, int rows, int64_t n, const int32_t* idx, double* out, int stride, const int32_t* perm,
                       cudaStream_t st) {
  if (n <= 0) return 0;
  gather_rows_kernel<<<nblk(n), 256, 0, st>>>(src, rows_total, row0, rows, n, idx, out, stride, perm);
  return 1;
}
int launch_flag_update(const DevState& s, int64_t n, const int32_t* idx, uint32_t and_mask, uint32_t or_mask, cudaStream_t st) {
  if (n <= 0) return 0;
  flag_update_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx, and_mask, or_mask);
  return 1;
}
int launch_gather_u32(const uint32_t* src, int64_t n, const int32_t* idx, uint32_t* out, const int32_t* perm, cudaStream_t st) {
  if (n <= 0) return 0;
  gather_u32_kernel<<<nblk(n), 256, 0, st>>>(src, n, idx, out, perm);
  return 1;
}
int launch_gather_u8(const uint8_t* src, int64_t n, const int32_t* idx, int32_t* out, const int32_t* perm, cudaStream_t st) {
  if (n <= 0) return 0;
  gather_u8_kernel<<<nblk(n), 256, 0, st>>>(src, n, idx, out, perm);
  return 1;
}
int launch_set_state_pos(const DevState& s, int64_t n, const int32_t* idx, const double* xyz, const double* hdg, cudaStream_t st) {
  if (n <= 0) return 0;
  set_state_pos_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx, xyz, hdg);
  return 1;
}
int launch_respawn(const DevState& s, const uint8_t* takeoff0, int64_t n, const int32_t* idx, const double* xyz, const double* hdg, cudaStream_t st) {
  if (n <= 0) return 0;
  respawn_kernel<<<nblk(n), 256, 0, st>>>(s, takeoff0, n, idx, xyz, hdg);
  return 1;
}
int launch_respawn_masked(const DevState& s, const uint8_t* takeoff0, const uint8_t* mask, const double* xyz, const double* hdg, cudaStream_t st) {
  if (s.n <= 0) return 0;
  respawn_masked_kernel<<<nblk(s.ld), 256, 0, st>>>(s, takeoff0, mask, xyz, hdg);  // s.ld is a whole number of warps
  return 1;
}
int launch_snapshot_save(const DevState& s, double* rows, uint32_t* flags, uint8_t* mode, cudaStream_t st) {
  if (s.n <= 0) return 0;
  snapshot_save_kernel<<<nblk(s.ld), 256, 0, st>>>(s, rows, flags, mode);
  return 1;
}
int launch_snapshot_restore(const DevState& s, const double* rows, const uint32_t* flags, const uint8_t* mode, int64_t n, const int32_t* idx,
                            const int32_t* src, cudaStream_t st) {
  if (n <= 0) return 0;
  snapshot_restore_kernel<<<nblk(n), 256, 0, st>>>(s, rows, flags, mode, n, idx, src);
  return 1;
}
int launch_snapshot_restore_masked(const DevState& s, const double* rows, const uint32_t* flags, const uint8_t* mode, const int32_t* src,
                                   cudaStream_t st) {
  if (s.n <= 0) return 0;
  snapshot_restore_masked_kernel<<<nblk(s.ld), 256, 0, st>>>(s, rows, flags, mode, src);  // s.ld is a whole number of warps
  return 1;
}
int launch_stash_vprev(const DevState& s, int64_t n, const int32_t* idx, cudaStream_t st) {
  if (n <= 0) return 0;
  stash_vprev_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx);
  return 1;
}
int launch_gather_vprev(const DevState& s, int64_t n, const int32_t* idx, double* out, cudaStream_t st) {
  if (n <= 0) return 0;
  gather_vprev_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx, out);
  return 1;
}
int launch_reset_pid(const DevState& s, int64_t n, const int32_t* idx, int pid0, int n_pids, cudaStream_t st) {
  if (n <= 0) return 0;
  reset_pid_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx, pid0, n_pids);
  return 1;
}
int launch_gather_xyz(const double* xyz, int64_t n, const int32_t* idx, double* out, cudaStream_t st) {
  if (n <= 0) return 0;
  gather_xyz_kernel<<<nblk(n), 256, 0, st>>>(xyz, n, idx, out);
  return 1;
}
int launch_tracker_cmd(const DevState& s, int64_t n, const int32_t* idx, const double* rows, cudaStream_t st) {
  if (n <= 0) return 0;
  tracker_cmd_kernel<<<nblk(n), 256, 0, st>>>(s, n, idx, rows);
  return 1;
}
int launch_set_geom(double* geom, int64_t n, const int32_t* idx, int64_t offset, const int32_t* pset, const DevParams* params, cudaStream_t st) {
  if (n <= 0) return 0;
  set_geom_kernel<<<nblk(n), 256, 0, st>>>(geom, n, idx, offset, pset, params);
  return 1;
}
int launch_set_pset(int32_t* pset, int64_t n, const int32_t* idx, int64_t offset, const int32_t* values, cudaStream_t st) {
  if (n <= 0) return 0;
  set_pset_kernel<<<nblk(n), 256, 0, st>>>(pset, n, idx, offset, values);
  return 1;
}
