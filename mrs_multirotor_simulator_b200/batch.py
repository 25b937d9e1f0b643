"""UavBatch — host-side mirror of the reference's UavSystem API for a whole batch of UAVs.

Thin numpy wrapper over the C ABI (include/mrsb.h); every method forwards to one mrsb_* entry
point, which cites the reference member it replaces.  Arrays are row-per-UAV; 3x3 matrices are 9
doubles column-major like the reference's internal ODE state (multirotor_model.hpp:204-214).
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import MAX_MOTORS, ControllerParams, CreateInfo, DeviceView, ModelParams, check

(INPUT_UNKNOWN, ACTUATOR_CMD, CONTROL_GROUP_CMD, ATTITUDE_RATE_CMD, ATTITUDE_CMD, TILT_HDG_RATE_CMD,
 ACCELERATION_HDG_RATE_CMD, ACCELERATION_HDG_CMD, VELOCITY_HDG_RATE_CMD, VELOCITY_HDG_CMD, POSITION_CMD) = range(11)

STRIDE = {ACTUATOR_CMD: MAX_MOTORS, CONTROL_GROUP_CMD: 4, ATTITUDE_RATE_CMD: 4, ATTITUDE_CMD: 10, TILT_HDG_RATE_CMD: 5,
          ACCELERATION_HDG_RATE_CMD: 4, ACCELERATION_HDG_CMD: 4, VELOCITY_HDG_RATE_CMD: 4, VELOCITY_HDG_CMD: 4, POSITION_CMD: 4}


def model_params(d):
    """Airframe dict (airframes.py) or ModelParams -> ModelParams, with J and the allocation
    scaling derived by the library (mrsb_model_params_finalize: uav_system_ros.cpp:98-103, 664-671)."""
    if isinstance(d, ModelParams):
        return d
    p = ModelParams()
    n = int(d["n_motors"])
    p.n_motors = n
    p.ground_enabled = int(bool(d.get("ground_enabled", False)))
    p.takeoff_patch_enabled = int(bool(d.get("takeoff_patch_enabled", False)))
    p.g = float(d.get("g", 9.81))
    for k in ("mass", "kf", "km", "prop_radius", "arm_length", "body_height", "motor_time_constant", "max_rpm", "min_rpm",
              "air_resistance_coeff"):
        setattr(p, k, float(d[k]))
    p.ground_z = float(d.get("ground_z", 0.0))
    A = np.asarray(d["allocation"], dtype=np.float64).reshape(4, n)
    for r in range(4):
        for m in range(n):
            p.allocation_matrix[r * MAX_MOTORS + m] = float(A[r, m])
    _lib.lib().mrsb_model_params_finalize(C.byref(p))
    if d.get("J") is not None:
        J = np.asarray(d["J"], dtype=np.float64).reshape(3, 3)
        for r in range(3):
            for c in range(3):
                p.J[3 * r + c] = float(J[r, c])
    return p


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _idx(idx):
    return None if idx is None else np.ascontiguousarray(idx, dtype=np.int32)


class UavBatch:
    """A shard of UAVs resident on one GPU: `UavSystem(params, spawn_pos, spawn_heading)` for each
    (uav_system.hpp:144-153)."""

    def __init__(self, types, type_of_uav=None, spawn_xyz=None, spawn_heading=None, n=None, device=0, n_global=None, shard_begin=0):
        L = _lib.lib()
        self._L = L
        self.types = [model_params(t) for t in types]
        arr = (ModelParams * len(self.types))(*self.types)
        if n is None:
            if spawn_xyz is not None:
                n = len(np.asarray(spawn_xyz).reshape(-1, 3))
            elif type_of_uav is not None and n_global is None:
                n = len(type_of_uav)
            else:
                n = 1
        self.n = int(n)
        self.n_global = int(n_global) if n_global is not None else self.n
        self.shard_begin = int(shard_begin)
        tou = None if type_of_uav is None else np.ascontiguousarray(type_of_uav, dtype=np.int32)
        if tou is not None and len(tou) != self.n_global:
            raise ValueError("type_of_uav must have n_global entries")
        xyz = None if spawn_xyz is None else np.ascontiguousarray(spawn_xyz, dtype=np.float64).reshape(self.n, 3)
        hdg = None if spawn_heading is None else np.ascontiguousarray(spawn_heading, dtype=np.float64).reshape(self.n)
        info = CreateInfo(device=device, n_types=len(self.types), types=arr, n_local=self.n, n_global=self.n_global, shard_begin=self.shard_begin,
                          type_of_uav=_ptr(tou), spawn_xyz=_ptr(xyz), spawn_heading=_ptr(hdg))
        h = C.c_void_p()
        check(L.mrsb_create(C.byref(info), C.byref(h)))
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self._L.mrsb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _n(self, idx):
        return self.n if idx is None else len(idx)

    # ---- commands (UavSystem::setInput, uav_system.hpp:175-248) ---------------------------------
    def set_input(self, mode, payload=None, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        if mode == INPUT_UNKNOWN:
            check(self._L.mrsb_clear_input(self.h, n, _ptr(idx)))
            return
        pl = np.ascontiguousarray(payload, dtype=np.float64).reshape(n, -1)
        if mode == ACTUATOR_CMD and pl.shape[1] < MAX_MOTORS:
            pl = np.ascontiguousarray(np.pad(pl, ((0, 0), (0, MAX_MOTORS - pl.shape[1]))))
        if pl.shape[1] != STRIDE[mode]:
            raise ValueError(f"mode {mode} needs rows of {STRIDE[mode]} doubles, got {pl.shape[1]}")
        check(self._L.mrsb_set_input(self.h, mode, n, _ptr(idx), _ptr(pl), pl.shape[1]))

    def set_input_device(self, mode, payload_ptr, stride, n=None, idx_ptr=None):
        """payload_ptr / idx_ptr: raw device addresses (e.g. torch tensor .data_ptr())."""
        check(self._L.mrsb_set_input_device(self.h, mode, self.n if n is None else n, idx_ptr, payload_ptr, stride))

    def set_input_async(self, mode, payload_ptr, stride):
        """Whole-batch setInput from host rows at address `payload_ptr` (pinned), uploaded on its own stream."""
        check(self._L.mrsb_set_input_async(self.h, mode, payload_ptr, stride))

    def get_positions_async(self, out_ptr):
        """Positions [n][3] -> host address `out_ptr` (pinned), downloaded on its own stream; valid after sync()."""
        check(self._L.mrsb_get_positions_async(self.h, out_ptr))

    def set_input_rows_async(self, n, idx_ptr, modes_ptr, payload_ptr, stride):
        """Row k sets UAV idx[k] to input mode modes[k] with payload row k, k < n, a later row for the same UAV winning: host
        addresses (pinned) of int32 idx [n], int32 modes [n] and float64 rows [n][stride], uploaded on the upload stream; they
        must stay untouched until sync()."""
        check(self._L.mrsb_set_input_rows_async(self.h, int(n), idx_ptr, modes_ptr, payload_ptr, int(stride)))

    def get_observations_async(self, out_ptr):
        """odometry 13 | IMU acceleration 3 | range 1 of the position subset (all UAVs without one) -> host address `out_ptr`
        (pinned, [m][17]), downloaded on the download stream; valid after sync()."""
        check(self._L.mrsb_get_observations_async(self.h, out_ptr))

    def set_position_subset(self, idx=None):
        """The UAVs get_positions_async and get_observations_async deliver from now on (None: all)."""
        idx = _idx(idx)
        check(self._L.mrsb_set_position_subset(self.h, 0 if idx is None else len(idx), _ptr(idx)))

    def set_feedforward(self, kind, payload, idx=None):
        """kind: 'acceleration_hdg_rate' | 'acceleration_hdg' | 'velocity_hdg' | 'velocity_hdg_rate' (uav_system.hpp:254-272)."""
        idx = _idx(idx)
        n = self._n(idx)
        pl = np.ascontiguousarray(payload, dtype=np.float64).reshape(n, 4)
        check(getattr(self._L, "mrsb_set_feedforward_" + kind)(self.h, n, _ptr(idx), _ptr(pl)))

    def set_tracker_cmd(self, rows, idx=None):
        """UavSystemRos::callbackTrackerCmd (uav_system_ros.cpp:987-1022): rows [n][11] = velocity xyz, acceleration xyz,
        heading_rate, use_velocity_horizontal, use_velocity_vertical, use_heading_rate, use_acceleration."""
        idx = _idx(idx)
        n = self._n(idx)
        pl = np.ascontiguousarray(rows, dtype=np.float64).reshape(n, 11)
        check(self._L.mrsb_set_tracker_cmd(self.h, n, _ptr(idx), _ptr(pl)))

    def clear_feedforward(self, idx=None):
        idx = _idx(idx)
        check(self._L.mrsb_clear_feedforward(self.h, self._n(idx), _ptr(idx)))

    # ---- stepping -------------------------------------------------------------------------------
    def make_step(self, dt, k_substeps=1):
        check(self._L.mrsb_make_step(self.h, float(dt), int(k_substeps)))

    def run(self, dt, n_ticks, k_substeps=1, with_collisions=True):
        check(self._L.mrsb_run(self.h, float(dt), int(k_substeps), int(n_ticks), int(bool(with_collisions))))

    def set_iterate_without_input(self, enabled):
        """`iterate_without_input` of the reference (uav_system_ros.cpp:265): with False, UAVs without a command are not stepped."""
        check(self._L.mrsb_set_iterate_without_input(self.h, int(bool(enabled))))

    def set_outputs(self, imu=True, positions=True):
        """Which optional rows make_step stores: the fabricated accelerometer (multirotor_model.hpp:280-281) and the packed positions."""
        check(self._L.mrsb_set_outputs(self.h, (1 if imu else 0) | (2 if positions else 0)))

    def sync(self):
        check(self._L.mrsb_sync(self.h))

    @property
    def stream(self):
        return self._L.mrsb_get_stream(self.h)

    # ---- state ----------------------------------------------------------------------------------
    def get_state(self, idx=None, fields=("x", "v", "R", "omega", "motor_rpm")):
        idx = _idx(idx)
        n = self._n(idx)
        widths = {"x": 3, "v": 3, "R": 9, "omega": 3, "motor_rpm": MAX_MOTORS}
        out = {k: np.empty((n, widths[k])) for k in fields if k in widths}
        check(self._L.mrsb_get_state(self.h, n, _ptr(idx), *[_ptr(out.get(k)) for k in ("x", "v", "R", "omega", "motor_rpm")]))
        if "v_prev" in fields:
            out["v_prev"] = np.empty((n, 3))
            check(self._L.mrsb_get_v_prev(self.h, n, _ptr(idx), _ptr(out["v_prev"])))
        if "imu" in fields:
            out["imu"] = self.get_imu_acceleration(idx)
        return out

    def get_full_state(self, idx=None):
        return self.get_state(idx, ("x", "v", "R", "omega", "motor_rpm", "v_prev", "imu"))

    def get_imu_acceleration(self, idx=None):
        idx = _idx(idx)
        out = np.empty((self._n(idx), 3))
        check(self._L.mrsb_get_imu_acceleration(self.h, len(out), _ptr(idx), _ptr(out)))
        return out

    def set_state(self, idx=None, x=None, v=None, R=None, omega=None, motor_rpm=None):
        idx = _idx(idx)
        n = self._n(idx)
        arrs = [None if a is None else np.ascontiguousarray(a, dtype=np.float64).reshape(n, -1) for a in (x, v, R, omega, motor_rpm)]
        check(self._L.mrsb_set_state(self.h, n, _ptr(idx), *[_ptr(a) for a in arrs]))

    def set_state_pos(self, xyz, heading, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(n, 3)
        heading = np.ascontiguousarray(heading, dtype=np.float64).reshape(n)
        check(self._L.mrsb_set_state_pos(self.h, n, _ptr(idx), _ptr(xyz), _ptr(heading)))

    def respawn(self, xyz, heading, idx=None):
        """Episode reset: `UavSystem(params, pos, heading)` again for the addressed UAVs (uav_system.hpp:144-153), keeping their
        airframe, parameter edits and controller gains; see mrsb_respawn for what a fresh UAV holds."""
        idx = _idx(idx)
        n = self._n(idx)
        xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(n, 3)
        heading = np.ascontiguousarray(np.broadcast_to(heading, (n,)), dtype=np.float64)
        check(self._L.mrsb_respawn(self.h, n, _ptr(idx), _ptr(xyz), _ptr(heading)))

    def respawn_masked_device(self, mask_ptr, xyz_ptr, heading_ptr):
        """respawn() for every UAV i with mask[i] != 0, all three raw device addresses (e.g. torch tensor .data_ptr()): mask
        uint8 / bool [n], xyz float64 [n][3], heading float64 [n].  Enqueued on the handle's stream, no host synchronisation."""
        check(self._L.mrsb_respawn_masked_device(self.h, mask_ptr, xyz_ptr, heading_ptr))

    def snapshot(self):
        """A new Snapshot of this batch (709 bytes of device memory per UAV, nothing saved yet); see mrsb_snapshot_create for
        what it holds and what a restore keeps."""
        return Snapshot(self)

    def get_input_mode(self, idx=None):
        idx = _idx(idx)
        out = np.empty(self._n(idx), dtype=np.int32)
        check(self._L.mrsb_get_input_mode(self.h, len(out), _ptr(idx), _ptr(out)))
        return out

    def crash(self, idx=None):
        idx = _idx(idx)
        check(self._L.mrsb_crash(self.h, self._n(idx), _ptr(idx)))

    def has_crashed(self, idx=None):
        idx = _idx(idx)
        out = np.empty(self._n(idx), dtype=np.int32)
        check(self._L.mrsb_has_crashed(self.h, len(out), _ptr(idx), _ptr(out)))
        return out

    def apply_force(self, f, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        f = np.ascontiguousarray(f, dtype=np.float64).reshape(n, 3)
        check(self._L.mrsb_apply_force(self.h, n, _ptr(idx), _ptr(f)))

    def forces_written(self):
        """Call after writing ext_force through device_view(): the next collision pass then replaces every UAV's force."""
        check(self._L.mrsb_forces_written(self.h))

    def get_force(self, idx=None):
        idx = _idx(idx)
        out = np.empty((self._n(idx), 3))
        check(self._L.mrsb_get_external_force(self.h, len(out), _ptr(idx), _ptr(out)))
        return out

    def set_external_moment(self, m, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        m = np.ascontiguousarray(m, dtype=np.float64).reshape(n, 3)
        check(self._L.mrsb_set_external_moment(self.h, n, _ptr(idx), _ptr(m)))

    # ---- parameters -----------------------------------------------------------------------------
    def get_params(self, uav=0):
        p = ModelParams()
        check(self._L.mrsb_get_params(self.h, uav, C.byref(p)))
        return p

    def set_params(self, params, idx=None):
        idx = _idx(idx)
        p = model_params(params)
        check(self._L.mrsb_set_params(self.h, self._n(idx), _ptr(idx), C.byref(p)))

    def get_controller_params(self, uav=0):
        p = ControllerParams()
        check(self._L.mrsb_get_controller_params(self.h, uav, C.byref(p)))
        return p

    def set_controller_params(self, which, values, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        v = [float(x) for x in np.atleast_1d(values)]
        if which == "mixer":
            check(self._L.mrsb_set_mixer_params(self.h, n, _ptr(idx), int(v[0] != 0)))
        else:
            fn = getattr(self._L, f"mrsb_set_{which}_controller_params")
            check(fn(self.h, n, _ptr(idx), *v))

    def get_mixer_allocation(self, uav=0):
        out = np.zeros((MAX_MOTORS, 4))
        check(self._L.mrsb_get_mixer_allocation(self.h, uav, _ptr(out)))
        return out

    # ---- the ROS wrapper's arithmetic around the path (uav_system_ros.cpp) -------------------------
    def timeout_input(self, idx=None):
        """UavSystemRos::timeoutInput (uav_system_ros.cpp:474-647): the active command becomes its hover version."""
        idx = _idx(idx)
        check(self._L.mrsb_timeout_input(self.h, self._n(idx), _ptr(idx)))

    def _rows(self, fn, width, idx):
        idx = _idx(idx)
        out = np.empty((self._n(idx), width))
        check(getattr(self._L, fn)(self.h, len(out), _ptr(idx), _ptr(out)))
        return out

    def get_odometry(self, idx=None):
        """rows [13]: position, orientation xyzw, body-frame linear velocity, angular velocity (uav_system_ros.cpp:340-368)."""
        return self._rows("mrsb_get_odometry", 13, idx)

    def get_imu(self, idx=None):
        """rows [10]: angular velocity, linear acceleration, orientation xyzw (uav_system_ros.cpp:374-395)."""
        return self._rows("mrsb_get_imu", 10, idx)

    def get_rangefinder(self, idx=None):
        """rows [1]: down-looking range (uav_system_ros.cpp:401-420)."""
        return self._rows("mrsb_get_rangefinder", 1, idx)

    def pack_observations_device(self, out_ptr, stride=17):
        """odometry 13 | IMU acceleration 3 | range 1 for every UAV into a device buffer (no host round trip)."""
        check(self._L.mrsb_pack_observations_device(self.h, out_ptr, stride))

    def pack_neighbours_device(self, radius, k, idx_ptr=None, rows_ptr=None, count_ptr=None, stride=None):
        """The k nearest UAVs within `radius` of every UAV, by (d2, index), into device buffers (raw addresses, e.g. torch tensor
        .data_ptr(); any may be None, not all): indices int32 [n][k] (-1 past the last), rows float64 [n][stride >= 6k] of
        [x_j - x_i | v_j - v_i] per neighbour (zero past the last), counts int32 [n] (not capped by k).  No host round trip."""
        check(self._L.mrsb_pack_neighbours_device(self.h, float(radius), int(k), idx_ptr, rows_ptr, 6 * int(k) if stride is None else int(stride),
                                                  count_ptr))

    def set_mass(self, mass, idx=None):
        idx = _idx(idx)
        m = np.ascontiguousarray(np.broadcast_to(mass, (self._n(idx),)), dtype=np.float64)
        check(self._L.mrsb_set_mass(self.h, len(m), _ptr(idx), _ptr(m)))

    def set_ground_z(self, z, idx=None):
        idx = _idx(idx)
        z = np.ascontiguousarray(np.broadcast_to(z, (self._n(idx),)), dtype=np.float64)
        check(self._L.mrsb_set_ground_z(self.h, len(z), _ptr(idx), _ptr(z)))

    # ---- collisions -----------------------------------------------------------------------------
    def set_collisions(self, enabled, crash, rebounce):
        check(self._L.mrsb_set_collisions(self.h, int(bool(enabled)), int(bool(crash)), float(rebounce)))

    def handle_collisions(self):
        check(self._L.mrsb_handle_collisions(self.h))

    def handle_collisions_gathered(self):
        check(self._L.mrsb_handle_collisions_gathered(self.h))

    def get_collision_pairs(self):
        """Directed pairs (i, j), global indices, sorted by (i, j), found by the last collision pass."""
        cnt = C.c_int64(0)
        check(self._L.mrsb_get_collision_pairs(self.h, None, 0, C.byref(cnt)))
        k = cnt.value
        pairs = np.zeros((max(k, 1), 2), dtype=np.int32)
        if k:
            check(self._L.mrsb_get_collision_pairs(self.h, _ptr(pairs), k, C.byref(cnt)))
        return pairs[:k]

    def set_pair_capacity(self, max_pairs):
        check(self._L.mrsb_set_pair_capacity(self.h, int(max_pairs)))

    def counters(self):
        out = np.zeros(5, dtype=np.int64)
        check(self._L.mrsb_get_counters(self.h, _ptr(out)))
        return dict(steps=int(out[0]), collision_passes=int(out[1]), pairs=int(out[2]), crashed=int(out[3]), launches=int(out[4]))

    def step_info(self):
        """Which stepping kernel the last make_step launched (diagnostics): variant 'direct' | 'staged', grid, motors, mode."""
        out = np.zeros(4, dtype=np.int32)
        check(self._L.mrsb_get_step_info(self.h, _ptr(out)))
        return dict(variant={0: "none", 1: "direct", 2: "staged", 3: "staged+peer-stores"}[int(out[0])], grid=int(out[1]), n_motors=int(out[2]),
                    mode=int(out[3]))

    def sweep_launches(self):
        """Per airframe bucket: staged stepping launches that swept with alternating direction (diagnostics)."""
        out = np.zeros(8, dtype=np.int64)
        nb = C.c_int32()
        check(self._L.mrsb_get_sweep_launches(self.h, _ptr(out), len(out), C.byref(nb)))
        return out[: nb.value].tolist()

    def timeline(self, max_passes=4096):
        """Device-clock stamps of the last collision passes [k][8] (needs MRSB_TIMELINE=1 at creation); see mrsb_get_timeline."""
        out = np.zeros((max_passes, 8), dtype=np.uint64)
        n = C.c_int64(0)
        check(self._L.mrsb_get_timeline(self.h, _ptr(out), max_passes, C.byref(n)))
        return out[:n.value]

    def collision_info(self):
        """How the collision pass is organised on this handle (diagnostics; results do not depend on it)."""
        out = np.zeros(8, dtype=np.float64)
        check(self._L.mrsb_get_collision_info(self.h, _ptr(out)))
        return dict(cell=float(out[0]), neighbour_lists=bool(out[1]), list_radius=float(out[2]), skin=float(out[3]), passes=int(out[4]),
                    rebuilds=int(out[5]), crowded_uavs=int(out[6]), n_buckets=int(out[7]))

    # ---- sharded operation ----------------------------------------------------------------------
    @staticmethod
    def nccl_unique_id():
        buf = (C.c_char * 128)()
        check(_lib.lib().mrsb_nccl_unique_id(buf))
        return bytes(buf)

    def comm_init_nccl(self, n_ranks, rank, unique_id):
        buf = (C.c_char * 128).from_buffer_copy(unique_id)
        check(self._L.mrsb_comm_init_nccl(self.h, n_ranks, rank, buf))

    def exchange_mode(self):
        """0 single shard, 1 NCCL all-gather per tick, 2 pull over peer memory (hand-shake + halo fetch over NVLink)."""
        return int(self._L.mrsb_exchange_mode(self.h))

    def gather_buffer(self):
        p = C.c_void_p()
        nbytes = C.c_size_t()
        check(self._L.mrsb_gather_buffer(self.h, C.byref(p), C.byref(nbytes)))
        return p.value, nbytes.value

    def publish_positions(self):
        check(self._L.mrsb_publish_positions(self.h))

    def device_view(self):
        v = DeviceView()
        check(self._L.mrsb_get_device_view(self.h, C.byref(v)))
        return v


class Snapshot:
    """The full dynamic state of every UAV of a UavBatch (mrsb_snapshot_*): state, motors, PIDs, command, feed-forwards, forces,
    v_prev, flags and input mode.  A restore keeps each UAV's airframe, parameters, gains and collision geometry, as respawn does."""

    def __init__(self, batch):
        self.batch = batch
        sid = C.c_int32(0)
        check(batch._L.mrsb_snapshot_create(batch.h, C.byref(sid)))
        self.id = sid.value

    def save(self):
        """Save every UAV's state; enqueued on the batch's stream, no host synchronisation."""
        check(self.batch._L.mrsb_snapshot_save(self.batch.h, self.id))

    def restore(self, idx=None, src=None):
        """UAV idx[k] (None: every UAV) takes the saved record src[k] (None: its own)."""
        idx = _idx(idx)
        src = _idx(src)
        n = self.batch.n if idx is None and src is None else len(idx if idx is not None else src)
        check(self.batch._L.mrsb_snapshot_restore(self.batch.h, self.id, n, _ptr(idx), _ptr(src)))

    def restore_device(self, src_ptr=None):
        """UAV e takes the saved record src[e] where 0 <= src[e] < n and is left alone elsewhere; src_ptr is a raw device address
        of int32 [n] (e.g. torch tensor .data_ptr()), None: every UAV takes its own.  Enqueued on the batch's stream, no host
        synchronisation."""
        check(self.batch._L.mrsb_snapshot_restore_device(self.batch.h, self.id, src_ptr))

    def to_bytes(self):
        """Host image of the snapshot (header + device bytes) for load_bytes() on a handle of the same shard, e.g. in another process."""
        size = C.c_size_t(0)
        check(self.batch._L.mrsb_snapshot_image_size(self.batch.h, C.byref(size)))
        buf = np.empty(size.value, dtype=np.uint8)
        check(self.batch._L.mrsb_snapshot_download(self.batch.h, self.id, _ptr(buf), size.value))
        return buf.tobytes()

    def load_bytes(self, b):
        buf = np.frombuffer(b, dtype=np.uint8)
        check(self.batch._L.mrsb_snapshot_upload(self.batch.h, self.id, _ptr(buf), len(buf)))

    def free(self):
        if self.id is not None and getattr(self.batch, "h", None):
            check(self.batch._L.mrsb_snapshot_free(self.batch.h, self.id))
        self.id = None
