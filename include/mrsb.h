/*
 * mrsb.h — C ABI of libmrsb: batched multirotor stepping on NVIDIA B200 (sm_100a).
 *
 * One handle owns ONE batch ("shard") of UAVs resident on ONE CUDA device.  Every entry point
 * below replaces a member of the reference's per-UAV, CPU-only classes; the reference member is
 * cited as file:line relative to the reference repository root, with
 *   US  = include/mrs_multirotor_simulator/uav_system/uav_system.hpp
 *   MM  = include/mrs_multirotor_simulator/uav_system/multirotor_model.hpp
 *   CTL = include/mrs_multirotor_simulator/uav_system/controllers
 *   SIM = src/multirotor_simulator.cpp
 *   ROSW= src/uav_system_ros.cpp
 *
 * Conventions
 *  - plain pointers and sizes only; no C++/torch types cross this boundary;
 *  - every function returns MRSB_OK (0) or a negative mrsb_status; mrsb_last_error() has the text;
 *  - `idx` arguments select UAVs of THIS handle (local indices 0..n_local-1); idx == NULL means
 *    "UAVs 0..n-1 in order" (so n == n_local addresses the whole batch);
 *  - payload arrays are row-per-UAV ("AoS") in HOST memory unless the function name ends in
 *    `_device`; the library transposes to its structure-of-arrays device layout;
 *  - 3x3 matrices (R, orientation) are packed COLUMN-major, 9 doubles, exactly like the
 *    reference packs R into its ODE state (MM:204-214);
 *  - all work is enqueued on the handle's CUDA stream; getters synchronise that stream, nothing
 *    else does (use mrsb_sync);
 *  - a handle is driven by one host thread at a time (the reference serialises with a mutex,
 *    ROSW:267).
 *  - there is NO CPU fallback: without a CUDA device mrsb_create fails with MRSB_ERR_CUDA.
 */
#ifndef MRSB_H
#define MRSB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRSB_VERSION_MAJOR 0
#define MRSB_VERSION_MINOR 1

#define MRSB_MAX_MOTORS 8 /* largest shipped airframe: naki, config/uavs/naki.yaml (8 motors) */

typedef struct mrsb_sim* mrsb_handle;

typedef enum mrsb_status {
  MRSB_OK             = 0,
  MRSB_ERR_INVALID    = -1, /* bad argument (NULL, out-of-range index, n_motors > MRSB_MAX_MOTORS …) */
  MRSB_ERR_CUDA       = -2, /* CUDA runtime failure, or no device */
  MRSB_ERR_NCCL       = -3, /* NCCL failure or libnccl not loadable */
  MRSB_ERR_CAPACITY   = -4, /* caller buffer too small (count is still reported) */
  MRSB_ERR_STATE      = -5  /* call not valid in the current state (e.g. comm not initialised) */
} mrsb_status;

/* INPUT_MODE, same numeric values as UavSystem::INPUT_MODE (US:19-32). */
typedef enum mrsb_input_mode {
  MRSB_INPUT_UNKNOWN           = 0,
  MRSB_ACTUATOR_CMD            = 1,
  MRSB_CONTROL_GROUP_CMD       = 2,
  MRSB_ATTITUDE_RATE_CMD       = 3,
  MRSB_ATTITUDE_CMD            = 4,
  MRSB_TILT_HDG_RATE_CMD       = 5,
  MRSB_ACCELERATION_HDG_RATE_CMD = 6,
  MRSB_ACCELERATION_HDG_CMD    = 7,
  MRSB_VELOCITY_HDG_RATE_CMD   = 8,
  MRSB_VELOCITY_HDG_CMD        = 9,
  MRSB_POSITION_CMD            = 10
} mrsb_input_mode;

/* MultirotorModel::ModelParams (MM:24-88).  J and allocation_matrix are ROW-major here:
 * J(r,c) = J[3*r+c]; allocation_matrix(r,m) = allocation_matrix[r*MRSB_MAX_MOTORS+m], r=0..3
 * (torque x, torque y, torque z, thrust), columns m >= n_motors are ignored.  The allocation
 * matrix is the already-scaled one (rows *= arm*kf, arm*kf, km*3*prop_radius*kf, kf: MM:59-62,
 * ROSW:100-103).  mrsb_model_params_default() and mrsb_model_params_finalize() do that scaling. */
typedef struct mrsb_model_params {
  int32_t n_motors;
  int32_t ground_enabled;        /* MM:84  */
  int32_t takeoff_patch_enabled; /* MM:87 — initial value of the per-UAV one-way flag (MM:275) */
  int32_t reserved_;
  double  g;
  double  mass;
  double  kf;
  double  km;
  double  prop_radius;
  double  arm_length;
  double  body_height;
  double  motor_time_constant;
  double  max_rpm;
  double  min_rpm;
  double  air_resistance_coeff;
  double  ground_z;
  double  J[9];
  double  allocation_matrix[4 * MRSB_MAX_MOTORS];
} mrsb_model_params;

/* Controller gains: Mixer::Params (CTL/mixer.hpp:13-16), RateController::Params
 * (CTL/rate_controller.hpp:15-20), AttitudeController::Params (CTL/attitude_controller.hpp:14-21),
 * VelocityController::Params (CTL/velocity_controller.hpp:14-20), PositionController::Params
 * (CTL/position_controller.hpp:13-20). */
typedef struct mrsb_controller_params {
  int32_t mixer_desaturation;
  int32_t reserved_;
  double  rate_kp, rate_kd, rate_ki;
  double  att_kp, att_kd, att_ki, att_max_rate_roll_pitch, att_max_rate_yaw;
  double  vel_kp, vel_kd, vel_ki, vel_max_acceleration;
  double  pos_kp, pos_kd, pos_ki, pos_max_velocity;
} mrsb_controller_params;

/* Everything needed to build a batch.  One entry of `types` is one airframe; `type_of_uav`
 * assigns an airframe to every UAV.
 *
 * Sharding (SURVEY §8e): a multi-GPU job runs one handle per GPU.  n_global is the swarm size,
 * [shard_begin, shard_begin+n_local) the contiguous global index range this handle owns.  For a
 * single-GPU job n_global == n_local and shard_begin == 0.  `type_of_uav` has n_global entries
 * (airframe geometry and mass of REMOTE UAVs are needed by the collision pass, SIM:342,350);
 * spawn arrays have n_local entries. */
typedef struct mrsb_create_info {
  int32_t                  device;        /* CUDA device ordinal */
  int32_t                  n_types;
  const mrsb_model_params* types;         /* [n_types] */
  int64_t                  n_local;
  int64_t                  n_global;
  int64_t                  shard_begin;
  const int32_t*           type_of_uav;   /* [n_global], NULL = all type 0 */
  const double*            spawn_xyz;     /* [n_local*3], NULL = origin */
  const double*            spawn_heading; /* [n_local],   NULL = 0 */
} mrsb_create_info;

/* ---- library ---------------------------------------------------------------------------- */
const char* mrsb_last_error(void);
int         mrsb_version(void); /* major*1000 + minor */

/* x500 defaults of ModelParams::ModelParams() (MM:26-66), allocation already scaled. */
void mrsb_model_params_default(mrsb_model_params* out);
/* Derive J (ROSW:664-671) and scale an UNSCALED allocation matrix in place (ROSW:98-103). */
void mrsb_model_params_finalize(mrsb_model_params* p);
/* Header defaults of the five controller Params classes (same as config/controllers/ yaml). */
void mrsb_controller_params_default(mrsb_controller_params* out);
/* Mixer::calculateAllocation (CTL/mixer.hpp:72-101) for an airframe, no handle needed: normalised
 * pseudo-inverse of the allocation matrix, row-major [n_motors][4] in out[MRSB_MAX_MOTORS*4]. */
void mrsb_mixer_allocation_of(const mrsb_model_params* params, double* out);

/* How mrsb_create lays out a batch (pure host computation, no device needed).  A batch with 2..8 airframe types present is stored
 * bucketed: its UAVs sorted stably by type, every type padded to whole tiles of 128 slots, so that each tile of the device
 * arrays holds one airframe.  type_of_local_uav[n]: type of every local UAV.  Outputs (any may be NULL except n_slots):
 * slot_of_uav[n], *n_slots (a multiple of 128), bucket_first_slot[n_types] (-1: type absent or batch not bucketed) and
 * bucket_count[n_types].  Returns the number of buckets (1 = not bucketed: slot_of_uav[i] = i) or a negative mrsb_status. */
int mrsb_bucket_layout(int64_t n, int32_t n_types, const int32_t* type_of_local_uav, int32_t* slot_of_uav, int64_t* n_slots, int64_t* bucket_first_slot,
                       int64_t* bucket_count);

/* ---- lifetime: UavSystem(params, spawn_pos, spawn_heading) for every UAV (US:144-153) ----- */
int mrsb_create(const mrsb_create_info* info, mrsb_handle* out);
int mrsb_destroy(mrsb_handle h);
int mrsb_sync(mrsb_handle h);
int64_t mrsb_n_local(mrsb_handle h);
int64_t mrsb_n_global(mrsb_handle h);
/* The CUDA stream (cudaStream_t) all work of this handle is enqueued on. */
void* mrsb_get_stream(mrsb_handle h);

/* ---- commands: UavSystem::setInput overloads (US:175-248) ----------------------------------
 * payload row layouts (doubles):
 *   actuators            [MRSB_MAX_MOTORS] motors 0..n_motors-1, rest ignored (CTL/references.hpp:15-27)
 *   control_group        [4] roll pitch yaw throttle                          (:33-59)
 *   attitude_rate        [4] rate_x rate_y rate_z throttle                    (:65-91)
 *   attitude             [10] orientation (col-major 3x3), throttle           (:97-114)
 *   tilt_hdg_rate        [5] tilt_vector xyz, heading_rate, throttle          (:120-139)
 *   acceleration_hdg_rate[4] acceleration xyz, heading_rate                   (:145-164)
 *   acceleration_hdg     [4] acceleration xyz, heading                        (:170-192)
 *   velocity_hdg_rate    [4] velocity xyz, heading_rate                       (:198-220)
 *   velocity_hdg         [4] velocity xyz, heading                            (:226-248)
 *   position             [4] position xyz, heading                            (:254-271)        */
int mrsb_set_input_actuators(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_input_control_group(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_input_attitude_rate(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_input_attitude(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_input_tilt_hdg_rate(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_input_acceleration_hdg_rate(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_input_acceleration_hdg(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_input_velocity_hdg_rate(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_input_velocity_hdg(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_input_position(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
/* UavSystem::setInput(void) (US:245-248): mode := INPUT_UNKNOWN (motors driven to zero). */
int mrsb_clear_input(mrsb_handle h, int64_t n, const int32_t* idx);
/* Generic form of the ten setters above; `mode` is an mrsb_input_mode, `stride` the row length. */
int mrsb_set_input(mrsb_handle h, int32_t mode, int64_t n, const int32_t* idx, const double* payload, int32_t stride);
/* Same, but idx/payload are DEVICE pointers valid on the handle's device; no host round trip. */
int mrsb_set_input_device(mrsb_handle h, int32_t mode, int64_t n, const int32_t* idx_dev, const double* payload_dev, int32_t stride);

/* Pipelined variants for host loops that feed commands and read poses EVERY tick (the reference
 * node does both: ROS command callbacks in, publishPoses out, SIM:215).  Both return at once:
 *  - mrsb_set_input_async: whole-batch setInput; the host rows (pinned memory recommended) are
 *    copied on a dedicated upload stream into one of two staging buffers while earlier ticks are
 *    still computing; the handle's stream waits for the copy before applying the command.  The
 *    caller must leave `payload` untouched until a later mrsb_sync / mrsb_wait_uploads.
 *  - mrsb_get_positions_async: snapshots the positions as of the work enqueued so far and copies
 *    them ([n_local][3] doubles) to `out_xyz` on a dedicated download stream while later ticks
 *    compute; `out_xyz` is valid after mrsb_sync (or mrsb_wait_downloads). */
int mrsb_set_input_async(mrsb_handle h, int32_t mode, const double* payload, int32_t stride);
int mrsb_get_positions_async(mrsb_handle h, double* out_xyz);
/* Pipelined sparse commands, for a node whose commands arrive one UAV at a time in any of the ten input modes (ROSW:679-981).
 * Row k sets UAV idx[k] to input mode modes[k] (1..10) with payload row payload[k*stride ...], exactly as if
 * mrsb_set_input(h, modes[k], 1, &idx[k], row k, stride) were called for k = 0..n-1 in order: a later row for the same UAV wins.
 * Host arrays, pinned recommended; they must stay untouched until mrsb_wait_uploads / mrsb_sync.  Returns at once: the arrays
 * go through the upload ring of mrsb_set_input_async (the two calls mix freely), and duplicates are resolved on the device.
 * Checked on the host before anything is enqueued (MRSB_ERR_INVALID, nothing changes): NULL arrays, n outside 0..INT32_MAX,
 * idx outside 0..n_local-1, mode 0 or outside 1..10, stride below the row length of any row's mode (actuator rows accept any
 * stride >= 1; motors past the stride get 0).  n == 0 is a no-op.  The batch stays single-mode (specialised stepping kernel,
 * cached tick graph) only if every row carries its mode; a later whole-batch call makes it single-mode again. */
int mrsb_set_input_rows_async(mrsb_handle h, int64_t n, const int32_t* idx, const int32_t* modes, const double* payload, int32_t stride);
/* Pipelined sensor rows (publishOdometry, publishIMU, publishRangefinder of every UAV's makeStep, ROSW:278-282): [m][17] =
 * odometry 13 | IMU linear acceleration 3 | range 1 (the rows of mrsb_pack_observations_device) of the work enqueued so far, for the
 * UAVs of mrsb_set_position_subset in its order (m = its n), or for all n_local UAVs.  Copied on the download stream with a
 * two-deep ring of its own; valid after mrsb_sync / mrsb_wait_downloads.  Either download call may be issued every tick, in any
 * order.  MRSB_ERR_STATE when the IMU rows are switched off (mrsb_set_outputs). */
int mrsb_get_observations_async(mrsb_handle h, double* out17);
/* The UAVs the async downloads deliver from now on: the n UAVs idx[] (out_xyz then holds [n][3], out17 [n][17], in idx order) — a
 * viewer that follows part of the swarm does not pay PCIe for all of it.  idx == NULL or n == 0: all of them again.  Synchronises. */
int mrsb_set_position_subset(mrsb_handle h, int64_t n, const int32_t* idx);
int mrsb_wait_uploads(mrsb_handle h);
int mrsb_wait_downloads(mrsb_handle h);

/* ---- feed-forwards: UavSystem::setFeedforward overloads (US:254-272); sticky, never cleared
 * by the reference (US:112-115).  Row layout [4]: xyz + heading or heading_rate.  mrsb_clear_
 * feedforward is an extension (the reference offers no way to unset the std::optional). */
int mrsb_set_feedforward_acceleration_hdg_rate(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_feedforward_acceleration_hdg(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_feedforward_velocity_hdg(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
int mrsb_set_feedforward_velocity_hdg_rate(mrsb_handle h, int64_t n, const int32_t* idx, const double* payload);
/* UavSystemRos::callbackTrackerCmd (src/uav_system_ros.cpp:987-1022): one mrs_msgs::TrackerCommand per UAV
 * becomes all four feed-forwards — VelocityHdg(v, 0), VelocityHdgRate(v, heading_rate), AccelerationHdg(a, 0),
 * AccelerationHdgRate(a, heading_rate) — where the parts the message does not "use" are zero.
 * rows[k][11] = velocity xyz | acceleration xyz | heading_rate | use_velocity_horizontal |
 * use_velocity_vertical | use_heading_rate | use_acceleration (flags: non-zero = true). */
#define MRSB_TRACKER_CMD_STRIDE 11
int mrsb_set_tracker_cmd(mrsb_handle h, int64_t n, const int32_t* idx, const double* rows);
int mrsb_clear_feedforward(mrsb_handle h, int64_t n, const int32_t* idx);

/* ---- stepping: UavSystem::makeStep(dt) (US:304-380) for every UAV of the batch -------------
 * k_substeps >= 1 consecutive makeStep(dt) calls are fused into one kernel launch with the UAV
 * state held in registers in between (commands and external force are constant over them,
 * exactly as k back-to-back reference calls with no setInput/applyForce in between). */
int mrsb_make_step(mrsb_handle h, double dt, int32_t k_substeps);

/* One tick of the reference node's loop (SIM:198-231): makeStep for all, then handleCollisions;
 * repeated n_ticks times without host synchronisation (with neighbour lists each tick is ONE CUDA
 * graph launch: stepping kernel + collision pass).  In a sharded job every rank must call it with
 * the same arguments (the collision pass contains the cross-shard exchange). */
int mrsb_run(mrsb_handle h, double dt, int32_t k_substeps, int32_t n_ticks, int32_t with_collisions);

/* UavSystemRos::makeStep (ROSW:242-271) steps a UAV only `if (_iterate_without_input_ || time_last_input_ > 0)`
 * (ROSW:265; parameter `iterate_without_input`, config/multirotor_simulator.yaml:10, default true).  With enabled = 0 a
 * UAV that has not received a command yet (any mrsb_set_input* with a payload), or whose input timed out
 * (mrsb_timeout_input resets time_last_input_, ROSW:256-259), is left untouched by mrsb_make_step: state, PIDs, IMU and
 * flags keep their values. */
int mrsb_set_iterate_without_input(mrsb_handle h, int32_t enabled);

/* Which optional per-UAV rows mrsb_make_step stores (default: all).  The fabricated accelerometer (MM:280-281) and the packed
 * positions cost 24 bytes per UAV-step each; a caller that never reads them (RL loops reading state through the device view)
 * switches them off.  With MRSB_OUT_IMU off, mrsb_get_imu_acceleration / mrsb_get_imu / mrsb_pack_observations_device fail with
 * MRSB_ERR_STATE instead of returning stale values.  The library keeps storing positions whenever the collision pass or a
 * peer shard needs them, whatever the mask says. */
#define MRSB_OUT_IMU 1u
#define MRSB_OUT_POSITIONS 2u
int mrsb_set_outputs(mrsb_handle h, uint32_t mask);

/* ---- state: UavSystem::getState (US:386-390, MM:90-98), getImuAcceleration (US:424-427) ----
 * any output pointer may be NULL.  Rows: x[3] v[3] R[9 col-major] omega[3] motor_rpm[MRSB_MAX_MOTORS]. */
int mrsb_get_state(mrsb_handle h, int64_t n, const int32_t* idx, double* x, double* v, double* R, double* omega, double* motor_rpm);
int mrsb_get_v_prev(mrsb_handle h, int64_t n, const int32_t* idx, double* v_prev);
int mrsb_get_imu_acceleration(mrsb_handle h, int64_t n, const int32_t* idx, double* acc);
/* MultirotorModel::setState (MM:424-433): x, v, R, omega, motor_rpm; NULL = leave unchanged. */
int mrsb_set_state(mrsb_handle h, int64_t n, const int32_t* idx, const double* x, const double* v, const double* R, const double* omega, const double* motor_rpm);
/* MultirotorModel::setStatePos (MM:439-446): x := pos, initial_pos := pos, R := Rz(-heading). */
int mrsb_set_state_pos(mrsb_handle h, int64_t n, const int32_t* idx, const double* xyz, const double* heading);
/* Episode reset.  UavSystem(params, spawn_pos, spawn_heading) (US:144-153) again for the n UAVs idx[] (NULL: 0..n-1), keeping
 * their airframe, parameter edits (mrsb_set_params / mrsb_set_mass / mrsb_set_ground_z) and controller gains; xyz[n][3],
 * heading[n] in host memory.  Afterwards each of them is exactly a freshly created UAV with those parameters and gains:
 *   x = xyz, spawn z = xyz.z, R = Rz(-heading) (as mrsb_set_state_pos); v = omega = 0, motor RPM = 0, IMU acceleration = 0,
 *   v_prev = v; all twelve PIDs zero; input mode INPUT_UNKNOWN with no command ever received (with iterate_without_input
 *   off it stays frozen until its next command, ROSW:265); no feed-forwards; zero external force and moment; not crashed.
 * The take-off patch flag (MM:87, MM:275) gets the value of the UAV's parameter set, i.e. the one given at mrsb_create or by the
 * last mrsb_set_params (mrsb_set_mass / mrsb_set_ground_z keep it): a UAV respawned on the ground gets the one-way patch
 * again, as a newly spawned one would.  (A reference user who rebuilt a UavSystem from getParams() after take-off would pass
 * the consumed flag instead.)  The ROS wrapper's two warm-up steps (ROSW:223-232) are not part of UavSystem and not done.
 * Local to this shard (not collective); may be issued anywhere between two collision passes.  n == 0 is a no-op; duplicate
 * indices are undefined, as with every setter. */
int mrsb_respawn(mrsb_handle h, int64_t n, const int32_t* idx, const double* xyz, const double* heading);
/* Same for every local UAV i with mask_dev[i] != 0 (uint8, n_local entries: a torch.bool tensor works as is); xyz_dev[n_local][3]
 * and heading_dev[n_local] are DEVICE arrays, read only where the mask is set.  Enqueued on the handle's stream; no host
 * synchronisation, no host round trip; the host never learns whether anybody was respawned.  A mask with a bit set makes the
 * next collision pass rebuild its table (on every rank of a pull-exchange run); an all-zero mask changes nothing.  The batch
 * counts as mixed-mode afterwards: an RL loop sets its commands for the whole batch next (mrsb_set_input_device with
 * idx_dev == NULL), which keeps the stepping kernel specialised for that mode. */
int mrsb_respawn_masked_device(mrsb_handle h, const uint8_t* mask_dev, const double* xyz_dev, const double* heading_dev);

/* ---- snapshots: save and restore every UAV's full dynamic state (checkpoint / resume, branching rollouts) ----
 * MultirotorModel::setState (MM:424-433) puts back x, v, R, omega and motor RPM only; v_prev, the twelve PIDs, the active
 * command, the feed-forwards and the take-off flag of a UavSystem (US:16-118 members) cannot be set from outside.  A snapshot
 * holds all of it for every local UAV of one handle, as one record per UAV in external (caller) order, whatever the bucketing:
 *   88 doubles — x, v, R (column-major), omega [18] | motor RPM [8] | PID last errors [12] and integrals [12] | command payload
 *   [10] and cached cos/sin of its heading [2] | the four feed-forwards [13] | external force [3] | external moment [3] | IMU
 *   acceleration [3] | v_prev [3] | spawn z [1] — plus a uint32 of flags (crashed, take-off patch, v_prev, feed-forwards, had a
 *   command) and the uint8 INPUT_MODE: 709 bytes per UAV (743 MB of device memory at 1 Mi UAVs).
 * Restoring a UAV puts back its record and nothing else.  Like a respawn, it keeps the UAV's airframe, parameter set
 * (mrsb_set_params / mrsb_set_mass / mrsb_set_ground_z and the gain setters keep the values they set) and collision geometry;
 * handle-level options (collisions, iterate_without_input, outputs, position subset) are not part of a snapshot either.  This is
 * deliberate: parameters stay host-side bookkeeping, which a restore on the device could not update without a synchronisation.
 * The integrals of the rate PIDs are not stored while rate ki == 0; they are zero then (every change of ki resets them), so a
 * record saved with ki == 0 restores them as zero.  A record copied between UAVs of different motor counts is copied
 * verbatim: defined, but not the continuation of any flight.
 * Save and restore are local to this shard (not collective) and may be issued anywhere between two collision passes.  A
 * restore makes the next collision pass rebuild its neighbour table (on every rank of a pull-exchange run) and replace every
 * UAV's external force.  Afterwards the batch counts as single-mode if every UAV took its own record (src NULL: the mode it
 * had at the save) or if it had, at the save and now, the same single mode; otherwise as mixed-mode.  The RL order (restore,
 * then commands for the whole batch, then step) keeps the specialised stepping kernel either way. */

/* A snapshot of this handle's UAVs (709 bytes per UAV of device memory; nothing saved yet).  It belongs to the handle:
 * mrsb_snapshot_free or, at the latest, mrsb_destroy releases it.  Unknown or freed ids are MRSB_ERR_INVALID everywhere. */
int mrsb_snapshot_create(mrsb_handle h, int32_t* id);
int mrsb_snapshot_free(mrsb_handle h, int32_t id);
/* Save the state of every local UAV into snapshot `id` (replacing what it held).  Enqueued on the handle's stream, no host
 * synchronisation; changes nothing in the simulation (no displacement word, graph or counter but the launch counter).  It
 * records the batch's input-mode and external-moment hints of the moment. */
int mrsb_snapshot_save(mrsb_handle h, int32_t id);
/* Host form: UAV idx[k] (idx NULL: UAV k) takes saved record src[k] (src NULL: its own), k < n.  Indices and records outside
 * 0..n_local-1 are MRSB_ERR_INVALID; n == 0 is a no-op; duplicate idx entries are undefined.  MRSB_ERR_STATE if the snapshot was
 * never saved or uploaded. */
int mrsb_snapshot_restore(mrsb_handle h, int32_t id, int64_t n, const int32_t* idx, const int32_t* src);
/* Device form, per UAV: src_dev[e] (int32, n_local entries, DEVICE memory) in 0..n_local-1 makes UAV e take that record; any
 * other value leaves UAV e untouched.  src_dev NULL: every UAV takes its own record.  Enqueued on the handle's stream; no host
 * synchronisation, no host round trip. */
int mrsb_snapshot_restore_device(mrsb_handle h, int32_t id, const int32_t* src_dev);
/* Host image of a snapshot, to resume in another process: a 48-byte header {char magic[8] "MRSBSNAP"; uint32 version, rows;
 * int64 n_local, n_global, shard_begin; int32 input-mode hint, external-moment hint} followed by the snapshot's device bytes
 * verbatim (rows [88][n_local] doubles, flags [n_local] uint32, mode [n_local] uint8).  *bytes = the image size of this handle.
 * download synchronises and needs exactly that many bytes; upload checks them, the magic, the version and that the image was made
 * by a handle of the same shard (n_local, n_global, shard_begin): MRSB_ERR_INVALID otherwise.  An uploaded snapshot restores as
 * a saved one. */
int mrsb_snapshot_image_size(mrsb_handle h, size_t* bytes);
int mrsb_snapshot_download(mrsb_handle h, int32_t id, void* host, size_t bytes);
int mrsb_snapshot_upload(mrsb_handle h, int32_t id, const void* host, size_t bytes);
/* Current INPUT_MODE of each UAV (US:95). */
int mrsb_get_input_mode(mrsb_handle h, int64_t n, const int32_t* idx, int32_t* mode);

/* UavSystem::crash / hasCrashed (US:278-289). */
int mrsb_crash(mrsb_handle h, int64_t n, const int32_t* idx);
int mrsb_has_crashed(mrsb_handle h, int64_t n, const int32_t* idx, int32_t* crashed);
/* UavSystem::applyForce (US:295-298, MM:292-295): external force [3] per UAV, held until replaced. */
int mrsb_apply_force(mrsb_handle h, int64_t n, const int32_t* idx, const double* force);
int mrsb_get_external_force(mrsb_handle h, int64_t n, const int32_t* idx, double* force);
/* MultirotorModel::setExternalMoment (MM:476-478). */
int mrsb_set_external_moment(mrsb_handle h, int64_t n, const int32_t* idx, const double* moment);

/* ---- parameters ----------------------------------------------------------------------------
 * UavSystem::getParams / setParams (US:395-409).  setParams re-creates all six controllers with
 * DEFAULT gains and resets their PIDs (US:404-409, 159-169) — reproduced.  The takeoff-patch flag
 * returned by get_params is the UAV's live one-way flag (MM:275). */
int mrsb_get_params(mrsb_handle h, int64_t uav, mrsb_model_params* out);
int mrsb_set_params(mrsb_handle h, int64_t n, const int32_t* idx, const mrsb_model_params* params);
/* set*ControllerParams (US:433-451): each resets that controller's PIDs (CTL setParams). */
int mrsb_set_mixer_params(mrsb_handle h, int64_t n, const int32_t* idx, int32_t desaturation);
int mrsb_set_rate_controller_params(mrsb_handle h, int64_t n, const int32_t* idx, double kp, double kd, double ki);
int mrsb_set_attitude_controller_params(mrsb_handle h, int64_t n, const int32_t* idx, double kp, double kd, double ki, double max_rate_roll_pitch, double max_rate_yaw);
int mrsb_set_velocity_controller_params(mrsb_handle h, int64_t n, const int32_t* idx, double kp, double kd, double ki, double max_acceleration);
int mrsb_set_position_controller_params(mrsb_handle h, int64_t n, const int32_t* idx, double kp, double kd, double ki, double max_velocity);
int mrsb_get_controller_params(mrsb_handle h, int64_t uav, mrsb_controller_params* out);
/* UavSystem::getMixerAllocation (US:415-418, CTL/mixer.hpp:72-101): normalised pseudo-inverse,
 * row-major [n_motors][4] written into out[MRSB_MAX_MOTORS*4]. */
int mrsb_get_mixer_allocation(mrsb_handle h, int64_t uav, double* out);

/* ---- the ROS wrapper's arithmetic around the path (src/uav_system_ros.cpp), batched -------------
 * mrsb_timeout_input: UavSystemRos::timeoutInput (ROSW:474-647) — replace the active command by its
 *   hover version (Position: hold the current position and heading; Velocity / Acceleration: zero;
 *   Attitude: level at the current heading, zero throttle; ...); the caller decides WHEN (the
 *   reference: no command for `input_timeout` seconds, ROSW:247-261).
 * mrsb_get_odometry:    publishOdometry (ROSW:340-368), rows [13]: position xyz, orientation
 *   quaternion xyzw (Eigen::Quaterniond(R)), linear velocity in the BODY frame (R^T v), angular velocity.
 * mrsb_get_imu:         publishIMU (ROSW:374-395), rows [10]: angular velocity, linear acceleration, orientation xyzw.
 * mrsb_get_rangefinder: publishRangefinder (ROSW:401-420), rows [1]: (z - ground_z)/cos(tilt) + 0.01, 41.0 beyond 40 m or when inverted.
 * mrsb_pack_observations_device: all of it for every UAV into a DEVICE buffer, rows [stride >= 17]:
 *   odometry 13 | IMU linear acceleration 3 | range 1 (enqueued on the handle's stream, no host round trip).
 * mrsb_set_mass / mrsb_set_ground_z: the set_mass / set_ground_z services (ROSW:1028-1080): like the
 *   reference they go through setParams, i.e. controllers return to default gains and PIDs reset. */
int mrsb_timeout_input(mrsb_handle h, int64_t n, const int32_t* idx);
int mrsb_get_odometry(mrsb_handle h, int64_t n, const int32_t* idx, double* out13);
int mrsb_get_imu(mrsb_handle h, int64_t n, const int32_t* idx, double* out10);
int mrsb_get_rangefinder(mrsb_handle h, int64_t n, const int32_t* idx, double* out1);
int mrsb_pack_observations_device(mrsb_handle h, double* out_dev, int32_t stride);
int mrsb_set_mass(mrsb_handle h, int64_t n, const int32_t* idx, const double* mass);
int mrsb_set_ground_z(mrsb_handle h, int64_t n, const int32_t* idx, const double* ground_z);

/* ---- neighbour observations (multi-agent RL) -------------------------------------------------
 * For every local UAV i, the UAVs j != i of this handle with d2 < radius*radius, where
 *   d2 = ((dx*dx) + dy*dy) + dz*dz,  dx = x_j - x_i (likewise y, z), in FP64 without contraction (the collision predicate's
 *   metric); radius*radius is rounded once, on the host, and the comparison is strict.
 * The set is sorted by (d2, j) ascending (ties go to the lower index) and its first min(count, k) are reported.  Crashed UAVs are
 * included (they are still bodies in the world).  A UAV with a non-finite position (NaN or Inf in any coordinate) has no
 * neighbours and is nobody's neighbour.
 * Outputs, all DEVICE arrays, any of them NULL but not all three:
 *   idx_dev[n_local][k]   neighbour indices (local = global on a single shard), -1 past the last neighbour;
 *   rows_dev              row i starts at i*stride (stride >= 6*k); block m of it = [x_j - x_i (3) | v_j - v_i (3)] in the world
 *                         frame, zero past the last neighbour; doubles past 6*k are not written (a caller can keep its own
 *                         observation columns beside them);
 *   count_dev[n_local]    how many UAVs are within the radius (not capped by k).
 * Positions and velocities are read from the state (mrsb_get_device_view's state rows 0-5), so the result is current right after
 * mrsb_set_state*, mrsb_respawn*, or a write through the device view, without mrsb_publish_positions, and also with
 * mrsb_set_outputs(h, 0) and collisions off.  Enqueued on the handle's stream; never synchronises the host.  Its workspace grows
 * on the first call for a batch size and is reused after that.  The collision pass' state (table, neighbour lists, pair list,
 * forces, counters [0-3]) is not touched; counter [4] counts the five kernels of a call.
 * Exact over the coordinate range |x|, |y|, |z| <= 2^30 * radius (beyond it the grid's cell arithmetic may leave out a true
 * neighbour; the table's reach exceeds the radius by a relative 2^-20 to absorb the rounding inside that range).
 * MRSB_ERR_INVALID: radius not finite or <= 0, k outside [1, MRSB_MAX_NEIGHBOURS], rows_dev with stride < 6*k, all outputs NULL.
 * MRSB_ERR_STATE: a sharded handle (n_global > n_local). */
#define MRSB_MAX_NEIGHBOURS 16
int mrsb_pack_neighbours_device(mrsb_handle h, double radius, int32_t k, int32_t* idx_dev, double* rows_dev, int32_t stride, int32_t* count_dev);

/* ---- collisions: MultirotorSimulator::handleCollisions (SIM:295-359) -----------------------
 * knobs = collisions/enabled, collisions/crash, collisions/rebounce (SIM:124-126,
 * cfg/multirotor_simulator.cfg:12-20).  The pass runs on the CURRENT positions: uniform-grid
 * spatial hash instead of the KD-tree, identical predicate (d2 < 3.0 && d2 < crit, nanoflann
 * L2 metric NF:452-486), so the directed pair list equals the reference's bit for bit. */
int mrsb_set_collisions(mrsb_handle h, int32_t enabled, int32_t crash, double rebounce);
int mrsb_handle_collisions(mrsb_handle h);
/* Directed pairs (i, j) — GLOBAL indices, i owned by this handle — found by the last pass,
 * sorted by (i, j).  ij holds up to cap pairs (2*cap int32).  *count receives the number found
 * (may exceed cap -> MRSB_ERR_CAPACITY). */
int mrsb_get_collision_pairs(mrsb_handle h, int32_t* ij, int64_t cap, int64_t* count);
/* Size of the device-side pair buffer (default max(4096, 4*n_local) pairs).  A pass that finds more
 * still applies every force / crash flag; only the recorded list is truncated and
 * mrsb_get_collision_pairs then reports MRSB_ERR_CAPACITY with the true count. */
int mrsb_set_pair_capacity(mrsb_handle h, int64_t max_pairs);
/* Cumulative counters since create: [0] steps, [1] collision passes, [2] directed pairs emitted
 * by the last pass, [3] crashed UAVs in this shard, [4] kernels launched by this handle. */
int mrsb_get_counters(mrsb_handle h, int64_t* out5);
/* Which stepping kernel the LAST mrsb_make_step launched (diagnostics; results do not depend on it — every variant
 * computes the same bits): [0] 0 = none yet, 1 = direct (one CTA per 128-UAV tile reading HBM), 2 = staged (persistent
 * CTAs, next tile fetched by TMA bulk copies into shared memory); [1] grid size; [2] motors per UAV the kernel was
 * specialised for (0 = per UAV); [3] INPUT_MODE it was specialised for (-1 = per UAV). */
int mrsb_get_step_info(mrsb_handle h, int32_t* out4);
/* Diagnostics: how many staged stepping launches of each airframe bucket swept with alternating direction (forward, backward,
 * forward, ...; results do not depend on it).  Only a handle with a single bucket alternates, and only launches that stream more
 * state than the L2 cache holds.  out[b] for the first min(cap, *n_buckets) buckets; synchronises the handle's stream. */
int mrsb_get_sweep_launches(mrsb_handle h, int64_t* out, int32_t cap, int32_t* n_buckets);
/* Diagnostics: device-clock stamps (nanoseconds, %globaltimer) the kernels of the last collision passes left when the handle was
 * created with the environment variable MRSB_TIMELINE=1: out[k][8] for the last min(n, max_passes, 4096) passes, oldest first —
 * [0] pass start, [1] peer hand-shake sent, [2] hand-shake complete, [3] halo refresh start, [4] list check start, [5] 1 if the pass
 * rebuilt its table, [6] unused, [7] list build start.  MRSB_ERR_STATE without the variable. */
int mrsb_get_timeline(mrsb_handle h, uint64_t* out, int64_t max_passes, int64_t* n_passes);
/* How the collision pass (SIM:295-359) is organised on this handle: [0] cell edge of the spatial hash in
 * metres, [1] 1 if neighbour lists are kept between table rebuilds (single-shard handles), [2] list
 * radius, [3] skin (the lists survive while twice the accumulated displacement bound stays below it),
 * [4] passes decided on the device, [5] of which rebuilt the table, [6] UAVs that had more candidates
 * than a list holds at the last rebuild (they walk the table's stencil instead), [7] buckets of the table.
 * Diagnostics only: pair lists, forces and crash flags do not depend on any of it. */
int mrsb_get_collision_info(mrsb_handle h, double* out8);

/* ---- sharded operation (one handle per GPU / process) --------------------------------------
 * A shard's collision pass needs the positions of the remote UAVs near its own.  With peer access
 * (mode 2 below) it fetches them itself; otherwise the exchange is ONE all-gather per collision
 * pass of the packed positions (n_global*3 doubles), provided in one of two ways:
 *  (a) in-library NCCL: rank 0 calls mrsb_nccl_unique_id, the caller ships the 128 bytes to all
 *      ranks (MPI, torch.distributed, a file …), every rank calls mrsb_comm_init_nccl;
 *  (b) caller-run collective: mrsb_gather_buffer returns the device pointer of the n_global*3
 *      buffer; before mrsb_handle_collisions_gathered() the caller all-gathers into it in place
 *      (this shard's slice, filled by mrsb_publish_positions, starts at shard_begin*3).        */
int mrsb_nccl_unique_id(void* out128);
int mrsb_comm_init_nccl(mrsb_handle h, int32_t n_ranks, int32_t rank, const void* unique_id128);
/* How mrsb_handle_collisions exchanges positions: 0 = single shard, 1 = NCCL all-gather of the
 * whole swarm every pass, 2 = pull over peer memory: every rank's position buffer (plus one bounding
 * box per 32 UAVs and the collision geometry) is mapped into its peers over CUDA IPC at
 * mrsb_comm_init_nccl; nothing is copied per tick — the pass' first kernel hand-shakes with the
 * peers, then reads exactly the remote positions it needs over NVLink (the candidates in its
 * neighbour lists; at a table rebuild the halo around its bounding box).  MRSB_NO_P2P=1 forces
 * mode 1.  In sharded runs every rank must issue the same sequence of mrsb_handle_collisions /
 * mrsb_run calls, as with any collective; any number of mrsb_make_step or state-writing calls may
 * lie between two passes.  Per-UAV model parameters that the collision pass of OTHER shards reads
 * (arm length, propeller radius, mass: mrsb_set_params, mrsb_set_mass) can be changed in mode 2
 * (peers read the owner's values) or on unsharded handles; in modes 0/1 of a sharded handle such a
 * call fails with MRSB_ERR_STATE. */
int mrsb_exchange_mode(mrsb_handle h);
int mrsb_gather_buffer(mrsb_handle h, void** device_ptr, size_t* bytes);
int mrsb_publish_positions(mrsb_handle h);
int mrsb_handle_collisions_gathered(mrsb_handle h);

/* ---- zero-copy access for device-resident callers (RL loops) -------------------------------
 * Device pointers into the library's tiled structure-of-arrays state.  Every per-UAV array is cut
 * into tiles of `tile` (=128) consecutive SLOTS; component c of the UAV in slot s of an array with R rows is at
 *     ptr[((s / tile) * R + c) * tile + s % tile].
 * A batch with one airframe type keeps UAV i in slot i (slot_of_uav == NULL).  A batch created with several types is
 * bucketed by type (every tile then holds one airframe, so the specialised kernels run): slot_of_uav[i] is the slot of
 * UAV i (device array of n_local int32).
 * state: R = state_rows = 18 (x 0-2, v 3-5, R column-major 6-14, omega 15-17 — the reference's
 * InternalState order, MM:204-214); motor_rpm: R = MRSB_MAX_MOTORS; imu_acc, ext_force: R = 3.
 * flags[i] bit 0 = crashed; input_mode[i] = INPUT_MODE.  Valid until mrsb_destroy. */
typedef struct mrsb_device_view {
  int32_t   tile;
  int32_t   state_rows;
  double*   state;
  double*   motor_rpm;
  double*   imu_acc;
  double*   ext_force;
  uint32_t* flags;
  uint8_t*  input_mode;
  const int32_t* slot_of_uav; /* NULL = identity */
} mrsb_device_view;
int mrsb_get_device_view(mrsb_handle h, mrsb_device_view* out);
/* After writing through the view: positions (state rows 0-2) -> mrsb_publish_positions, so that the
 * collision pass sees them; ext_force -> mrsb_forces_written, so that the next collision pass replaces
 * every UAV's force as MultirotorSimulator::handleCollisions does (SIM:356-358) and not only the ones it
 * last wrote itself.  mrsb_apply_force does this on its own. */
int mrsb_forces_written(mrsb_handle h);

/* ---- roofline denominators, measured on `device` (used by bench.py) --------------------------
 * FP64 FMA throughput in TFLOP/s (2 flop per FMA) and device-to-device copy bandwidth in GB/s
 * (read + write bytes). */
int mrsb_microbench_fp64(int device, double* tflops);
int mrsb_microbench_copy(int device, double* gbs);

#ifdef __cplusplus
}
#endif
#endif /* MRSB_H */
