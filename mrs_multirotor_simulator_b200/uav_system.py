"""UavSystem — drop-in mirror of mrs_multirotor_simulator::UavSystem (uav_system.hpp:16-118).

Same method names, argument meaning and error behaviour (none: bad numbers are clamped or zeroed
by the guards inside the stepping kernel, exactly like the reference) — but the object is a *view*
of one slot of a GPU-resident UavBatch, so a swarm of them steps in one kernel launch.

    ref (C++)                                   here (Python)
    UavSystem(params, spawn_pos, heading)       UavSystem(params, spawn_pos, heading)
    uav.setInput(reference::Position{...})      uav.setInput(Position(position=..., heading=...))
    uav.makeStep(dt)                            uav.makeStep(dt)
    uav.getState().x                            uav.getState().x

Command classes mirror controllers/references.hpp.
"""
from dataclasses import dataclass, field

import numpy as np

from . import batch as B


def _v3():
    return np.zeros(3)


@dataclass
class Actuators:  # references.hpp:15-27
    motors: np.ndarray = field(default_factory=lambda: np.zeros(0))


@dataclass
class ControlGroup:  # references.hpp:33-59
    roll: float = 0.0
    pitch: float = 0.0
    yaw: float = 0.0
    throttle: float = 0.0


@dataclass
class AttitudeRate:  # references.hpp:65-91
    rate_x: float = 0.0
    rate_y: float = 0.0
    rate_z: float = 0.0
    throttle: float = 0.0


@dataclass
class Attitude:  # references.hpp:97-114
    orientation: np.ndarray = field(default_factory=lambda: np.eye(3))
    throttle: float = 0.0


@dataclass
class TiltHdgRate:  # references.hpp:120-139
    tilt_vector: np.ndarray = field(default_factory=lambda: np.array([1.0, 0.0, 0.0]))
    heading_rate: float = 0.0
    throttle: float = 0.0


@dataclass
class AccelerationHdgRate:  # references.hpp:145-164
    acceleration: np.ndarray = field(default_factory=_v3)
    heading_rate: float = 0.0


@dataclass
class AccelerationHdg:  # references.hpp:170-192
    acceleration: np.ndarray = field(default_factory=_v3)
    heading: float = 0.0


@dataclass
class VelocityHdgRate:  # references.hpp:198-220
    velocity: np.ndarray = field(default_factory=_v3)
    heading_rate: float = 0.0


@dataclass
class VelocityHdg:  # references.hpp:226-248
    velocity: np.ndarray = field(default_factory=_v3)
    heading: float = 0.0


@dataclass
class Position:  # references.hpp:254-271
    position: np.ndarray = field(default_factory=_v3)
    heading: float = 0.0


@dataclass
class State:  # MultirotorModel::State, multirotor_model.hpp:90-98
    x: np.ndarray
    v: np.ndarray
    v_prev: np.ndarray
    R: np.ndarray  # 3x3
    omega: np.ndarray
    motor_rpm: np.ndarray  # n_motors


def _encode(cmd):
    if isinstance(cmd, Actuators):
        return B.ACTUATOR_CMD, np.asarray(cmd.motors, dtype=np.float64)
    if isinstance(cmd, ControlGroup):
        return B.CONTROL_GROUP_CMD, [cmd.roll, cmd.pitch, cmd.yaw, cmd.throttle]
    if isinstance(cmd, AttitudeRate):
        return B.ATTITUDE_RATE_CMD, [cmd.rate_x, cmd.rate_y, cmd.rate_z, cmd.throttle]
    if isinstance(cmd, Attitude):
        return B.ATTITUDE_CMD, list(np.asarray(cmd.orientation, dtype=np.float64).reshape(3, 3).T.reshape(9)) + [cmd.throttle]
    if isinstance(cmd, TiltHdgRate):
        return B.TILT_HDG_RATE_CMD, list(cmd.tilt_vector) + [cmd.heading_rate, cmd.throttle]
    if isinstance(cmd, AccelerationHdgRate):
        return B.ACCELERATION_HDG_RATE_CMD, list(cmd.acceleration) + [cmd.heading_rate]
    if isinstance(cmd, AccelerationHdg):
        return B.ACCELERATION_HDG_CMD, list(cmd.acceleration) + [cmd.heading]
    if isinstance(cmd, VelocityHdgRate):
        return B.VELOCITY_HDG_RATE_CMD, list(cmd.velocity) + [cmd.heading_rate]
    if isinstance(cmd, VelocityHdg):
        return B.VELOCITY_HDG_CMD, list(cmd.velocity) + [cmd.heading]
    if isinstance(cmd, Position):
        return B.POSITION_CMD, list(cmd.position) + [cmd.heading]
    raise TypeError(f"not a reference command: {type(cmd).__name__}")


class UavSystem:
    """One UAV.  Either owns a batch of one (`UavSystem(params, pos, heading)`) or is slot `index`
    of an existing batch (`UavSystem.view(batch, index)`); in the second form `makeStep` is not
    available per UAV — step the batch."""

    def __init__(self, model_params=None, spawn_pos=(0.0, 0.0, 0.0), spawn_heading=0.0, device=0):
        if model_params is None:
            p = B._lib.ModelParams()
            B._lib.lib().mrsb_model_params_default(p)  # header defaults (x500)
            model_params = p
        self._batch = B.UavBatch([model_params], spawn_xyz=[list(spawn_pos)], spawn_heading=[spawn_heading], n=1, device=device)
        self._i = 0
        self._owns = True

    @classmethod
    def view(cls, batch, index):
        self = cls.__new__(cls)
        self._batch, self._i, self._owns = batch, int(index), False
        return self

    @property
    def _idx(self):
        return [self._i]

    def respawn(self, spawn_pos=(0.0, 0.0, 0.0), spawn_heading=0.0):
        """Start over as `UavSystem(params, spawn_pos, spawn_heading)` (uav_system.hpp:144-153) with the current parameters and
        controller gains; the take-off patch flag is the one given at creation or by the last setParams (see mrsb_respawn)."""
        self._batch.respawn([list(spawn_pos)], [spawn_heading], self._idx)

    # uav_system.hpp:38
    def makeStep(self, dt):
        if not self._owns:
            raise RuntimeError("this UavSystem is a view of a batch: call batch.make_step(dt)")
        self._batch.make_step(dt, 1)

    # uav_system.hpp:40-43
    def crash(self):
        self._batch.crash(self._idx)

    def hasCrashed(self):
        return bool(self._batch.has_crashed(self._idx)[0])

    def applyForce(self, force):
        self._batch.apply_force([list(force)], self._idx)

    # uav_system.hpp:45-55
    def setInput(self, cmd=None):
        if cmd is None:
            self._batch.set_input(B.INPUT_UNKNOWN, None, self._idx)
            return
        mode, payload = _encode(cmd)
        self._batch.set_input(mode, [payload], self._idx)

    # uav_system.hpp:57-60
    def setFeedforward(self, cmd):
        kinds = {AccelerationHdgRate: "acceleration_hdg_rate", AccelerationHdg: "acceleration_hdg", VelocityHdg: "velocity_hdg",
                 VelocityHdgRate: "velocity_hdg_rate"}
        kind = kinds.get(type(cmd))
        if kind is None:
            raise TypeError("setFeedforward takes AccelerationHdgRate, AccelerationHdg, VelocityHdg or VelocityHdgRate")
        _, payload = _encode(cmd)
        self._batch.set_feedforward(kind, [payload], self._idx)

    # uav_system.hpp:62-67
    def getState(self):
        s = self._batch.get_state(self._idx, ("x", "v", "R", "omega", "motor_rpm", "v_prev"))
        n = self.getParams().n_motors
        return State(x=s["x"][0], v=s["v"][0], v_prev=s["v_prev"][0], R=s["R"][0].reshape(3, 3).T.copy(), omega=s["omega"][0],
                     motor_rpm=s["motor_rpm"][0][:n].copy())

    def getParams(self):
        return self._batch.get_params(self._i)

    def setParams(self, params):
        self._batch.set_params(params, self._idx)

    def getImuAcceleration(self):
        return self._batch.get_imu_acceleration(self._idx)[0]

    # uav_system.hpp:69-75
    def setMixerParams(self, desaturation=True):
        self._batch.set_controller_params("mixer", [float(desaturation)], self._idx)

    def setRateControllerParams(self, kp=4.0, kd=0.04, ki=0.0):
        self._batch.set_controller_params("rate", [kp, kd, ki], self._idx)

    def setAttitudeControllerParams(self, kp=6.0, kd=0.05, ki=0.01, max_rate_roll_pitch=10.0, max_rate_yaw=1.0):
        self._batch.set_controller_params("attitude", [kp, kd, ki, max_rate_roll_pitch, max_rate_yaw], self._idx)

    def setVelocityControllerParams(self, kp=2.0, kd=0.05, ki=0.01, max_acceleration=4.0):
        self._batch.set_controller_params("velocity", [kp, kd, ki, max_acceleration], self._idx)

    def setPositionControllerParams(self, kp=2.0, kd=0.15, ki=0.2, max_velocity=6.0):
        self._batch.set_controller_params("position", [kp, kd, ki, max_velocity], self._idx)

    def getMixerAllocation(self):
        n = self.getParams().n_motors
        return self._batch.get_mixer_allocation(self._i)[:n]
