// mrsb/uav_system.hpp — header-only C++ façade over the C ABI (include/mrsb.h).
//
// Source-level stand-in for mrs_multirotor_simulator::UavSystem (uav_system.hpp:16-118 of the
// reference): same method names, same argument meaning, value semantics for commands and state —
// but a UavSystem here is slot `i` of a GPU-resident mrsb::Swarm, so N of them step in one kernel
// launch (Swarm::makeStep) and the collision pass of the reference's node
// (multirotor_simulator.cpp:295-359) is Swarm::handleCollisions.  No Eigen: 3-vectors are
// std::array<double,3>, matrices std::array<double,9> in COLUMN-major order.
//
//   reference                                              this header
//   UavSystem uav(params, pos, heading);                   mrsb::Swarm swarm({params}, {}, {pos}, {heading}); auto uav = swarm[0];
//   uav.setInput(reference::Position{...});                uav.setInput(mrsb::reference::Position{...});
//   uav.makeStep(dt);                                      swarm.makeStep(dt);
//   uav.getState().x                                       uav.getState().x
#pragma once
#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../mrsb.h"

namespace mrsb {

using Vec3 = std::array<double, 3>;
using Mat3 = std::array<double, 9>;  // column-major

namespace reference {  // controllers/references.hpp:15-271
struct Actuators {
  std::vector<double> motors;
};
struct ControlGroup {
  double roll = 0, pitch = 0, yaw = 0, throttle = 0;
};
struct AttitudeRate {
  double rate_x = 0, rate_y = 0, rate_z = 0, throttle = 0;
};
struct Attitude {
  Mat3   orientation{1, 0, 0, 0, 1, 0, 0, 0, 1};
  double throttle = 0;
};
struct TiltHdgRate {
  Vec3   tilt_vector{1, 0, 0};
  double heading_rate = 0, throttle = 0;
};
struct AccelerationHdgRate {
  Vec3   acceleration{0, 0, 0};
  double heading_rate = 0;
};
struct AccelerationHdg {
  Vec3   acceleration{0, 0, 0};
  double heading = 0;
};
struct VelocityHdgRate {
  Vec3   velocity{0, 0, 0};
  double heading_rate = 0;
};
struct VelocityHdg {
  Vec3   velocity{0, 0, 0};
  double heading = 0;
};
struct Position {
  Vec3   position{0, 0, 0};
  double heading = 0;
};
}  // namespace reference

struct State {  // MultirotorModel::State, multirotor_model.hpp:90-98
  Vec3                x, v, v_prev, omega;
  Mat3                R;
  std::vector<double> motor_rpm;
};

inline void check(int rc) {
  if (rc != MRSB_OK) throw std::runtime_error(std::string("libmrsb: ") + mrsb_last_error());
}

inline mrsb_model_params defaultModelParams() {  // ModelParams::ModelParams(), x500
  mrsb_model_params p;
  mrsb_model_params_default(&p);
  return p;
}

class Swarm;

class UavSystem {
public:
  UavSystem(Swarm* swarm, int32_t index) : swarm_(swarm), i_(index) {}

  void crash();
  bool hasCrashed();
  void applyForce(const Vec3& force);

  void setInput(const reference::Actuators& c);
  void setInput(const reference::ControlGroup& c);
  void setInput(const reference::AttitudeRate& c);
  void setInput(const reference::Attitude& c);
  void setInput(const reference::TiltHdgRate& c);
  void setInput(const reference::AccelerationHdgRate& c);
  void setInput(const reference::AccelerationHdg& c);
  void setInput(const reference::VelocityHdgRate& c);
  void setInput(const reference::VelocityHdg& c);
  void setInput(const reference::Position& c);
  void setInput(void);

  void setFeedforward(const reference::AccelerationHdgRate& c);
  void setFeedforward(const reference::AccelerationHdg& c);
  void setFeedforward(const reference::VelocityHdg& c);
  void setFeedforward(const reference::VelocityHdgRate& c);

  State             getState(void);
  mrsb_model_params getParams(void);
  void              setParams(const mrsb_model_params& params);
  Vec3              getImuAcceleration(void);

  void setMixerParams(bool desaturation);
  void setRateControllerParams(double kp, double kd, double ki);
  void setAttitudeControllerParams(double kp, double kd, double ki, double max_rate_roll_pitch, double max_rate_yaw);
  void setVelocityControllerParams(double kp, double kd, double ki, double max_acceleration);
  void setPositionControllerParams(double kp, double kd, double ki, double max_velocity);

  std::vector<double> getMixerAllocation(void);  // row-major n_motors x 4

  // episode reset: UavSystem(params, pos, heading) again (uav_system.hpp:144-153), keeping parameters and gains (mrsb_respawn)
  void respawn(const Vec3& pos, double heading);

private:
  Swarm*  swarm_;
  int32_t i_;
};

class Swarm {
public:
  // one UavSystem(params, spawn_pos, spawn_heading) per entry of spawn_pos (uav_system.hpp:144-153)
  Swarm(const std::vector<mrsb_model_params>& types, const std::vector<int32_t>& type_of_uav, const std::vector<Vec3>& spawn_pos,
        const std::vector<double>& spawn_heading, int device = 0) {
    mrsb_create_info info{};
    info.device        = device;
    info.n_types       = int32_t(types.size());
    info.types         = types.data();
    info.n_local       = int64_t(spawn_pos.size());
    info.n_global      = info.n_local;
    info.shard_begin   = 0;
    info.type_of_uav   = type_of_uav.empty() ? nullptr : type_of_uav.data();
    info.spawn_xyz     = spawn_pos.empty() ? nullptr : spawn_pos.front().data();
    info.spawn_heading = spawn_heading.empty() ? nullptr : spawn_heading.data();
    check(mrsb_create(&info, &h_));
  }
  ~Swarm() { mrsb_destroy(h_); }
  Swarm(const Swarm&)            = delete;
  Swarm& operator=(const Swarm&) = delete;

  UavSystem operator[](int32_t i) { return UavSystem(this, i); }
  int64_t   size() const { return mrsb_n_local(h_); }

  // one tick of the reference node's loop (multirotor_simulator.cpp:211-217)
  void makeStep(double dt, int k_substeps = 1) { check(mrsb_make_step(h_, dt, k_substeps)); }
  void setCollisions(bool enabled, bool crash, double rebounce) { check(mrsb_set_collisions(h_, enabled, crash, rebounce)); }
  void handleCollisions() { check(mrsb_handle_collisions(h_)); }
  // n_ticks of makeStep + handleCollisions without host synchronisation (one CUDA graph launch per tick)
  void run(double dt, int n_ticks, int k_substeps = 1, bool with_collisions = true) { check(mrsb_run(h_, dt, k_substeps, n_ticks, with_collisions)); }
  // UavSystemRos::_iterate_without_input_ (uav_system_ros.cpp:52, 265)
  void setIterateWithoutInput(bool enabled) { check(mrsb_set_iterate_without_input(h_, enabled)); }
  // optional per-step rows: the fabricated accelerometer (multirotor_model.hpp:280-281) and the packed positions
  void setOutputs(bool imu, bool positions) { check(mrsb_set_outputs(h_, (imu ? MRSB_OUT_IMU : 0u) | (positions ? MRSB_OUT_POSITIONS : 0u))); }
  // ---- pipelined host I/O for a node loop (mrsb_*_async): every call returns at once; host arrays (pinned recommended) must stay
  // untouched until waitUploads / sync, results are valid after waitDownloads / sync
  // whole-batch command rows [size()][stride] of one mode
  void setInputAsync(int32_t mode, const double* payload, int32_t stride) { check(mrsb_set_input_async(h_, mode, payload, stride)); }
  // row k sets UAV idx[k] to mode modes[k] with payload row k, k < n; a later row for the same UAV wins
  void setInputRowsAsync(int64_t n, const int32_t* idx, const int32_t* modes, const double* payload, int32_t stride) {
    check(mrsb_set_input_rows_async(h_, n, idx, modes, payload, stride));
  }
  // positions [m][3] and odometry 13 | IMU acceleration 3 | range 1 rows [m][17] of the position subset (m = its size, else size())
  void getPositionsAsync(double* out_xyz) { check(mrsb_get_positions_async(h_, out_xyz)); }
  void getObservationsAsync(double* out17) { check(mrsb_get_observations_async(h_, out17)); }
  // the UAVs the async downloads deliver (idx == nullptr or n == 0: all of them)
  void setPositionSubset(int64_t n, const int32_t* idx) { check(mrsb_set_position_subset(h_, n, idx)); }
  void waitUploads() { check(mrsb_wait_uploads(h_)); }
  void waitDownloads() { check(mrsb_wait_downloads(h_)); }
  void sync() { check(mrsb_sync(h_)); }
  std::vector<std::array<int32_t, 2>> collisionPairs() {
    int64_t n = 0;
    check(mrsb_get_collision_pairs(h_, nullptr, 0, &n));
    std::vector<std::array<int32_t, 2>> out(static_cast<size_t>(n), std::array<int32_t, 2>{0, 0});
    if (n) check(mrsb_get_collision_pairs(h_, out.front().data(), n, &n));
    return out;
  }
  // after writing through mrsb_get_device_view: positions / external forces were changed behind the library's back
  void positionsWritten() { check(mrsb_publish_positions(h_)); }
  void forcesWritten() { check(mrsb_forces_written(h_)); }
  // episode reset of n UAVs (idx == nullptr: 0..n-1) at xyz[n][3], heading[n] (mrsb_respawn)
  void respawn(int64_t n, const int32_t* idx, const double* xyz, const double* heading) { check(mrsb_respawn(h_, n, idx, xyz, heading)); }
  // snapshots of every UAV's full state (mrsb_snapshot_*); a snapshot lives until snapshotFree or the Swarm's end
  int32_t snapshotCreate() {
    int32_t id = 0;
    check(mrsb_snapshot_create(h_, &id));
    return id;
  }
  void snapshotFree(int32_t id) { check(mrsb_snapshot_free(h_, id)); }
  void snapshotSave(int32_t id) { check(mrsb_snapshot_save(h_, id)); }
  // UAV idx[k] (idx == nullptr: k) takes saved record src[k] (src == nullptr: its own), k < n
  void snapshotRestore(int32_t id, int64_t n, const int32_t* idx = nullptr, const int32_t* src = nullptr) {
    check(mrsb_snapshot_restore(h_, id, n, idx, src));
  }
  void snapshotRestoreDevice(int32_t id, const int32_t* src_dev = nullptr) { check(mrsb_snapshot_restore_device(h_, id, src_dev)); }
  std::vector<unsigned char> snapshotImage(int32_t id) {
    size_t bytes = 0;
    check(mrsb_snapshot_image_size(h_, &bytes));
    std::vector<unsigned char> out(bytes);
    check(mrsb_snapshot_download(h_, id, out.data(), out.size()));
    return out;
  }
  void snapshotLoad(int32_t id, const std::vector<unsigned char>& image) { check(mrsb_snapshot_upload(h_, id, image.data(), image.size())); }
  mrsb_handle handle() { return h_; }

private:
  mrsb_handle h_ = nullptr;
};

// ---- UavSystem members ---------------------------------------------------------------------
inline void UavSystem::crash() { check(mrsb_crash(swarm_->handle(), 1, &i_)); }
inline bool UavSystem::hasCrashed() {
  int32_t c = 0;
  check(mrsb_has_crashed(swarm_->handle(), 1, &i_, &c));
  return c != 0;
}
inline void UavSystem::applyForce(const Vec3& f) { check(mrsb_apply_force(swarm_->handle(), 1, &i_, f.data())); }

inline void UavSystem::setInput(const reference::Actuators& c) {
  double p[MRSB_MAX_MOTORS] = {0};
  for (size_t m = 0; m < c.motors.size() && m < MRSB_MAX_MOTORS; m++) p[m] = c.motors[m];
  check(mrsb_set_input_actuators(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(const reference::ControlGroup& c) {
  const double p[4] = {c.roll, c.pitch, c.yaw, c.throttle};
  check(mrsb_set_input_control_group(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(const reference::AttitudeRate& c) {
  const double p[4] = {c.rate_x, c.rate_y, c.rate_z, c.throttle};
  check(mrsb_set_input_attitude_rate(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(const reference::Attitude& c) {
  double p[10];
  for (int k = 0; k < 9; k++) p[k] = c.orientation[k];
  p[9] = c.throttle;
  check(mrsb_set_input_attitude(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(const reference::TiltHdgRate& c) {
  const double p[5] = {c.tilt_vector[0], c.tilt_vector[1], c.tilt_vector[2], c.heading_rate, c.throttle};
  check(mrsb_set_input_tilt_hdg_rate(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(const reference::AccelerationHdgRate& c) {
  const double p[4] = {c.acceleration[0], c.acceleration[1], c.acceleration[2], c.heading_rate};
  check(mrsb_set_input_acceleration_hdg_rate(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(const reference::AccelerationHdg& c) {
  const double p[4] = {c.acceleration[0], c.acceleration[1], c.acceleration[2], c.heading};
  check(mrsb_set_input_acceleration_hdg(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(const reference::VelocityHdgRate& c) {
  const double p[4] = {c.velocity[0], c.velocity[1], c.velocity[2], c.heading_rate};
  check(mrsb_set_input_velocity_hdg_rate(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(const reference::VelocityHdg& c) {
  const double p[4] = {c.velocity[0], c.velocity[1], c.velocity[2], c.heading};
  check(mrsb_set_input_velocity_hdg(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(const reference::Position& c) {
  const double p[4] = {c.position[0], c.position[1], c.position[2], c.heading};
  check(mrsb_set_input_position(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setInput(void) { check(mrsb_clear_input(swarm_->handle(), 1, &i_)); }

inline void UavSystem::setFeedforward(const reference::AccelerationHdgRate& c) {
  const double p[4] = {c.acceleration[0], c.acceleration[1], c.acceleration[2], c.heading_rate};
  check(mrsb_set_feedforward_acceleration_hdg_rate(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setFeedforward(const reference::AccelerationHdg& c) {
  const double p[4] = {c.acceleration[0], c.acceleration[1], c.acceleration[2], c.heading};
  check(mrsb_set_feedforward_acceleration_hdg(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setFeedforward(const reference::VelocityHdg& c) {
  const double p[4] = {c.velocity[0], c.velocity[1], c.velocity[2], c.heading};
  check(mrsb_set_feedforward_velocity_hdg(swarm_->handle(), 1, &i_, p));
}
inline void UavSystem::setFeedforward(const reference::VelocityHdgRate& c) {
  const double p[4] = {c.velocity[0], c.velocity[1], c.velocity[2], c.heading_rate};
  check(mrsb_set_feedforward_velocity_hdg_rate(swarm_->handle(), 1, &i_, p));
}

inline State UavSystem::getState(void) {
  State  s;
  double rpm[MRSB_MAX_MOTORS];
  check(mrsb_get_state(swarm_->handle(), 1, &i_, s.x.data(), s.v.data(), s.R.data(), s.omega.data(), rpm));
  check(mrsb_get_v_prev(swarm_->handle(), 1, &i_, s.v_prev.data()));
  s.motor_rpm.assign(rpm, rpm + getParams().n_motors);
  return s;
}
inline mrsb_model_params UavSystem::getParams(void) {
  mrsb_model_params p;
  check(mrsb_get_params(swarm_->handle(), i_, &p));
  return p;
}
inline void UavSystem::setParams(const mrsb_model_params& params) { check(mrsb_set_params(swarm_->handle(), 1, &i_, &params)); }
inline Vec3 UavSystem::getImuAcceleration(void) {
  Vec3 a;
  check(mrsb_get_imu_acceleration(swarm_->handle(), 1, &i_, a.data()));
  return a;
}
inline void UavSystem::setMixerParams(bool desaturation) { check(mrsb_set_mixer_params(swarm_->handle(), 1, &i_, desaturation)); }
inline void UavSystem::setRateControllerParams(double kp, double kd, double ki) {
  check(mrsb_set_rate_controller_params(swarm_->handle(), 1, &i_, kp, kd, ki));
}
inline void UavSystem::setAttitudeControllerParams(double kp, double kd, double ki, double max_rate_roll_pitch, double max_rate_yaw) {
  check(mrsb_set_attitude_controller_params(swarm_->handle(), 1, &i_, kp, kd, ki, max_rate_roll_pitch, max_rate_yaw));
}
inline void UavSystem::setVelocityControllerParams(double kp, double kd, double ki, double max_acceleration) {
  check(mrsb_set_velocity_controller_params(swarm_->handle(), 1, &i_, kp, kd, ki, max_acceleration));
}
inline void UavSystem::setPositionControllerParams(double kp, double kd, double ki, double max_velocity) {
  check(mrsb_set_position_controller_params(swarm_->handle(), 1, &i_, kp, kd, ki, max_velocity));
}
inline std::vector<double> UavSystem::getMixerAllocation(void) {
  double m[MRSB_MAX_MOTORS * 4];
  check(mrsb_get_mixer_allocation(swarm_->handle(), i_, m));
  return std::vector<double>(m, m + 4 * getParams().n_motors);
}
inline void UavSystem::respawn(const Vec3& pos, double heading) { swarm_->respawn(1, &i_, pos.data(), &heading); }

}  // namespace mrsb
