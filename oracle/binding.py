"""ctypes binding of the CPU oracle (oracle/_build/liboracle.so, oracle/_ref/libref_nanoflann.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / ``--impl reference`` legs — never by the product package.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
MAX_MOTORS = 8

(INPUT_UNKNOWN, ACTUATOR_CMD, CONTROL_GROUP_CMD, ATTITUDE_RATE_CMD, ATTITUDE_CMD, TILT_HDG_RATE_CMD,
 ACCELERATION_HDG_RATE_CMD, ACCELERATION_HDG_CMD, VELOCITY_HDG_RATE_CMD, VELOCITY_HDG_CMD, POSITION_CMD) = range(11)

STRIDE = {ACTUATOR_CMD: 8, CONTROL_GROUP_CMD: 4, ATTITUDE_RATE_CMD: 4, ATTITUDE_CMD: 10, TILT_HDG_RATE_CMD: 5,
          ACCELERATION_HDG_RATE_CMD: 4, ACCELERATION_HDG_CMD: 4, VELOCITY_HDG_RATE_CMD: 4, VELOCITY_HDG_CMD: 4, POSITION_CMD: 4}


class OrcModelParams(C.Structure):
    _fields_ = [("n_motors", C.c_int32), ("ground_enabled", C.c_int32), ("takeoff_patch_enabled", C.c_int32), ("reserved_", C.c_int32),
                ("g", C.c_double), ("mass", C.c_double), ("kf", C.c_double), ("km", C.c_double), ("prop_radius", C.c_double),
                ("arm_length", C.c_double), ("body_height", C.c_double), ("motor_time_constant", C.c_double), ("max_rpm", C.c_double),
                ("min_rpm", C.c_double), ("air_resistance_coeff", C.c_double), ("ground_z", C.c_double), ("J", C.c_double * 9),
                ("allocation_matrix", C.c_double * (4 * MAX_MOTORS))]


COLLIDE_FN = C.CFUNCTYPE(C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_double, C.c_void_p, C.c_void_p,
                         C.c_void_p, C.c_int64, C.c_int32)

_lib = None
_ref = None


def build(fast=False):
    """(Re)build liboracle.so — and, when the reference tree is present, _ref/libref_nanoflann.so."""
    targets = ["all"] + (["fast"] if fast else [])
    subprocess.run(["make", "-s", "-C", HERE] + targets, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


def _bind_stepping(L):
    L.orc_create.restype = C.c_void_p
    L.orc_create.argtypes = [C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.orc_destroy.argtypes = [C.c_void_p]
    L.orc_set_input.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32]
    L.orc_set_feedforward.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]
    L.orc_make_step.argtypes = [C.c_void_p, C.c_double, C.c_int32, C.c_int32]
    L.orc_get_state.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 8
    L.orc_set_state.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 6
    L.orc_crash.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    L.orc_has_crashed.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.orc_apply_force.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.orc_get_force.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.orc_set_external_moment.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.orc_set_params.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.orc_get_params.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    L.orc_set_controller_params.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]
    L.orc_get_mixer_allocation.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    L.orc_get_pid_state.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    L.orc_pid_update.restype = C.c_double
    L.orc_pid_update.argtypes = [C.c_void_p] + [C.c_double] * 7
    L.orc_model_params_default.argtypes = [C.c_void_p]


_refsys = {}


def refsys_lib(flavour="default"):
    """The reference's own UavSystem compiled against oracle/shim (oracle/_ref); None if never built.
    flavour "default": the stand-in follows the same Eigen evaluation rules as uav_oracle.hpp;
    flavour "vec": the alternative reading (packet-ordered contiguous reductions, coefficient-based
    matrix x fixed-vector products) — used to measure how much an Eigen evaluation-order choice can matter."""
    if flavour not in _refsys:
        name = {"default": "libref_uavsystem.so", "vec": "libref_uavsystem_vec.so"}[flavour]
        path = os.path.join(HERE, "_ref", name)
        if not os.path.exists(path):
            return None
        L = C.CDLL(path)
        L.ref_uavsystem_flavour.restype = C.c_int32
        assert L.ref_uavsystem_flavour() == {"default": 1, "vec": 2}[flavour]
        _bind_stepping(L)
        _refsys[flavour] = L
    return _refsys[flavour]


def lib():
    global _lib
    if _lib is None:
        path = os.path.join(HERE, "_build", "liboracle.so")
        if not os.path.exists(path):
            build()
        L = C.CDLL(path)
        _bind_stepping(L)
        L.orc_handle_collisions.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
        L.orc_collide_port.restype = C.c_int64
        L.orc_collide_port.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_double, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_int64, C.c_int32]
        for name in ("orc_get_odometry", "orc_get_imu", "orc_get_rangefinder", "orc_set_mass", "orc_set_ground_z"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        L.orc_timeout_input.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        L.orc_u01.restype = C.c_double
        L.orc_u01.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64]
        _lib = L
    return _lib


_fast = None


def fast_lib():
    """liboracle_fast.so: the same restatement built -O3 -march=native ON THIS HOST (the flags depend on the CPU it runs on, so it
    is never shipped prebuilt) for the separately reported CPU-throughput figure; results may differ from the parity build in the
    last bits (FMA contraction).  None if it cannot be built here.  It is built in a temporary directory, so that the source
    tree may be read-only."""
    global _fast
    if _fast is None:
        try:
            with tempfile.TemporaryDirectory() as tmp:
                path = os.path.join(tmp, "liboracle_fast.so")
                subprocess.run(["make", "-s", "-B", "-C", HERE, "fast", f"FAST_OUT={path}"], check=True, stdout=subprocess.DEVNULL,
                               stderr=subprocess.DEVNULL, timeout=300)
                L = C.CDLL(path)  # stays mapped after the directory is removed
        except Exception:
            _fast = False
            return None
        _bind_stepping(L)
        L.orc_handle_collisions.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
        _fast = L
    return _fast or None


def ref_lib():
    """The real vendored nanoflann (oracle/_ref); None if it was never built."""
    global _ref
    if _ref is None:
        path = os.path.join(HERE, "_ref", "libref_nanoflann.so")
        if not os.path.exists(path):
            return None
        L = C.CDLL(path)
        L.ref_nanoflann_collide.restype = C.c_int64
        L.ref_nanoflann_collide.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_double, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_int64, C.c_int32]
        L.ref_nanoflann_count_neighbours.restype = C.c_int64
        L.ref_nanoflann_count_neighbours.argtypes = [C.c_int64, C.c_void_p]
        _ref = L
    return _ref


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _idx(idx):
    if idx is None:
        return None
    return np.ascontiguousarray(idx, dtype=np.int32)


def params_from_dict(d):
    """Airframe dict (see mrs_multirotor_simulator_b200.airframes) -> OrcModelParams.
    J as in ROSW:664-671, allocation scaling as in ROSW:98-103 / MM:59-62 (same operation order)."""
    p = OrcModelParams()
    n = int(d["n_motors"])
    p.n_motors = n
    p.ground_enabled = int(d.get("ground_enabled", False))
    p.takeoff_patch_enabled = int(d.get("takeoff_patch_enabled", False))
    p.g = float(d.get("g", 9.81))
    for k in ("mass", "kf", "km", "prop_radius", "arm_length", "body_height", "motor_time_constant", "max_rpm", "min_rpm",
              "air_resistance_coeff"):
        setattr(p, k, float(d[k]))
    p.ground_z = float(d.get("ground_z", 0.0))
    J = d.get("J")
    if J is None:
        m, a, bh = p.mass, p.arm_length, p.body_height
        J = [[m * (3.0 * a * a + bh * bh) / 12.0, 0, 0], [0, m * (3.0 * a * a + bh * bh) / 12.0, 0], [0, 0, (m * a * a) / 2.0]]
    for r in range(3):
        for c in range(3):
            p.J[3 * r + c] = float(J[r][c])
    A = np.array(d["allocation"], dtype=np.float64).reshape(4, n)
    scale = [p.arm_length * p.kf, p.arm_length * p.kf, p.km * (3.0 * p.prop_radius) * p.kf, p.kf]
    for r in range(4):
        for m_ in range(n):
            p.allocation_matrix[r * MAX_MOTORS + m_] = float(A[r, m_]) * scale[r]
    return p


def pid_update(state, kp, kd, ki, saturation, antiwindup, error, dt):
    """PIDController::update on state = np.array([last_error, integral]) (modified in place)."""
    return lib().orc_pid_update(_p(state), kp, kd, ki, saturation, antiwindup, error, dt)


def u01(seed, stream, index):
    """Vectorised counter RNG identical to orc_u01 (SURVEY §8d)."""
    with np.errstate(over="ignore"):
        g = np.uint64(0x9E3779B97F4A7C15)
        z = np.uint64(seed) + g * ((np.uint64(stream) << np.uint64(32)) + np.asarray(index, dtype=np.uint64))
        z = z + g
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


class OracleSwarm:
    """N independent restated UavSystems + the reference node's collision loop."""

    def _library(self):
        return lib()

    def __init__(self, types, type_of_uav=None, spawn_xyz=None, spawn_heading=None, n=None):
        L = self._L = self._library()
        self.types = [t if isinstance(t, OrcModelParams) else params_from_dict(t) for t in types]
        arr = (OrcModelParams * len(self.types))(*self.types)
        if n is None:
            n = len(type_of_uav) if type_of_uav is not None else (len(spawn_xyz) if spawn_xyz is not None else 1)
        self.n = int(n)
        tou = None if type_of_uav is None else np.ascontiguousarray(type_of_uav, dtype=np.int32)
        xyz = None if spawn_xyz is None else np.ascontiguousarray(spawn_xyz, dtype=np.float64).reshape(self.n, 3)
        hdg = None if spawn_heading is None else np.ascontiguousarray(spawn_heading, dtype=np.float64).reshape(self.n)
        self.h = L.orc_create(self.n, len(self.types), C.cast(arr, C.c_void_p), _p(tou), _p(xyz), _p(hdg))
        self.collisions = (0, 0, 0.0)

    def __del__(self):
        if getattr(self, "h", None):
            self._L.orc_destroy(self.h)
            self.h = None

    def _n(self, idx):
        return self.n if idx is None else len(idx)

    def set_input(self, mode, payload=None, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        if mode == INPUT_UNKNOWN:
            self._L.orc_set_input(self.h, mode, n, _p(idx), None, 0)
            return
        pl = np.ascontiguousarray(payload, dtype=np.float64).reshape(n, -1)
        if mode == ACTUATOR_CMD and pl.shape[1] < 8:
            pl = np.ascontiguousarray(np.pad(pl, ((0, 0), (0, 8 - pl.shape[1]))))
        assert pl.shape[1] == STRIDE[mode], (mode, pl.shape)
        self._L.orc_set_input(self.h, mode, n, _p(idx), _p(pl), pl.shape[1])

    def set_feedforward(self, kind, payload, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        pl = np.ascontiguousarray(payload, dtype=np.float64).reshape(n, 4)
        self._L.orc_set_feedforward(self.h, kind, n, _p(idx), _p(pl))

    def make_step(self, dt, n_steps=1, n_threads=1):
        self._L.orc_make_step(self.h, dt, n_steps, n_threads)

    def get_state(self, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        out = {"x": np.empty((n, 3)), "v": np.empty((n, 3)), "R": np.empty((n, 9)), "omega": np.empty((n, 3)), "motor_rpm": np.empty((n, 8)),
               "v_prev": np.empty((n, 3)), "imu": np.empty((n, 3))}
        self._L.orc_get_state(self.h, n, _p(idx), *[_p(out[k]) for k in ("x", "v", "R", "omega", "motor_rpm", "v_prev", "imu")])
        return out

    def set_state(self, idx=None, x=None, v=None, R=None, omega=None, motor_rpm=None):
        idx = _idx(idx)
        n = self._n(idx)
        arrs = [None if a is None else np.ascontiguousarray(a, dtype=np.float64).reshape(n, -1) for a in (x, v, R, omega, motor_rpm)]
        self._L.orc_set_state(self.h, n, _p(idx), *[_p(a) for a in arrs])

    def crash(self, idx=None):
        idx = _idx(idx)
        self._L.orc_crash(self.h, self._n(idx), _p(idx))

    def has_crashed(self, idx=None):
        idx = _idx(idx)
        out = np.zeros(self._n(idx), dtype=np.int32)
        self._L.orc_has_crashed(self.h, len(out), _p(idx), _p(out))
        return out

    def apply_force(self, f, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        f = np.ascontiguousarray(f, dtype=np.float64).reshape(n, 3)
        self._L.orc_apply_force(self.h, n, _p(idx), _p(f))

    def get_force(self, idx=None):
        idx = _idx(idx)
        out = np.empty((self._n(idx), 3))
        self._L.orc_get_force(self.h, len(out), _p(idx), _p(out))
        return out

    def set_external_moment(self, m, idx=None):
        idx = _idx(idx)
        n = self._n(idx)
        m = np.ascontiguousarray(m, dtype=np.float64).reshape(n, 3)
        self._L.orc_set_external_moment(self.h, n, _p(idx), _p(m))

    def set_params(self, params, idx=None):
        idx = _idx(idx)
        p = params if isinstance(params, OrcModelParams) else params_from_dict(params)
        self._L.orc_set_params(self.h, self._n(idx), _p(idx), C.byref(p))

    def get_params(self, uav):
        p = OrcModelParams()
        self._L.orc_get_params(self.h, uav, C.byref(p))
        return p

    def set_controller_params(self, which, values, idx=None):
        idx = _idx(idx)
        v = np.ascontiguousarray(values, dtype=np.float64)
        self._L.orc_set_controller_params(self.h, {"mixer": 0, "rate": 1, "attitude": 2, "velocity": 3, "position": 4}[which], self._n(idx), _p(idx), _p(v))

    def get_mixer_allocation(self, uav=0):
        out = np.zeros((8, 4))
        self._L.orc_get_mixer_allocation(self.h, uav, _p(out))
        return out

    def get_pid_state(self, uav=0):
        out = np.zeros(24)
        self._L.orc_get_pid_state(self.h, uav, _p(out))
        return out

    def timeout_input(self, idx=None):
        idx = _idx(idx)
        self._L.orc_timeout_input(self.h, self._n(idx), _p(idx))

    def _rows(self, fn, width, idx):
        idx = _idx(idx)
        out = np.empty((self._n(idx), width))
        getattr(self._L, fn)(self.h, len(out), _p(idx), _p(out))
        return out

    def get_odometry(self, idx=None):
        return self._rows("orc_get_odometry", 13, idx)

    def get_imu(self, idx=None):
        return self._rows("orc_get_imu", 10, idx)

    def get_rangefinder(self, idx=None):
        return self._rows("orc_get_rangefinder", 1, idx)

    def set_mass(self, mass, idx=None):
        idx = _idx(idx)
        m = np.ascontiguousarray(np.broadcast_to(mass, (self._n(idx),)), dtype=np.float64)
        self._L.orc_set_mass(self.h, len(m), _p(idx), _p(m))

    def set_ground_z(self, z, idx=None):
        idx = _idx(idx)
        z = np.ascontiguousarray(np.broadcast_to(z, (self._n(idx),)), dtype=np.float64)
        self._L.orc_set_ground_z(self.h, len(z), _p(idx), _p(z))

    def set_collisions(self, enabled, crash, rebounce):
        self.collisions = (int(enabled), int(crash), float(rebounce))

    def handle_collisions(self, engine="port", n_threads=1, cap=1 << 20):
        """Returns the directed pair list (k,2) in evaluation order."""
        fn = None
        if engine == "nanoflann":
            R = ref_lib()
            if R is None:
                raise RuntimeError("oracle/_ref/libref_nanoflann.so not built")
            fn = C.cast(R.ref_nanoflann_collide, C.c_void_p)
        pairs = np.zeros((cap, 2), dtype=np.int32)
        cnt = C.c_int64(0)
        en, cr, rb = self.collisions
        self._L.orc_handle_collisions(self.h, en, cr, rb, fn, n_threads, _p(pairs), cap, C.byref(cnt))
        return pairs[:min(cnt.value, cap)].copy()


class FastOracleSwarm(OracleSwarm):
    """OracleSwarm on the -O3 -march=native build (throughput figure only, never a parity reference)."""

    def _library(self):
        L = fast_lib()
        if L is None:
            raise RuntimeError("liboracle_fast.so cannot be built on this host")
        return L


class RefSwarm(OracleSwarm):
    """N UavSystems of the reference's OWN source, compiled here against the Eigen/odeint stand-ins
    (oracle/_ref/libref_uavsystem*.so, see oracle/ref_uavsystem.cpp).  Same harness as OracleSwarm;
    stepping only — collisions, timeout synthesis and the ROS-wrapper rows are not part of UavSystem."""

    def __init__(self, *a, flavour="default", **kw):
        self._flavour = flavour
        super().__init__(*a, **kw)

    def _library(self):
        L = refsys_lib(self._flavour)
        if L is None:
            raise RuntimeError("oracle/_ref/libref_uavsystem*.so not built (needs the reference tree: make -C oracle refsys)")
        return L

    def handle_collisions(self, *a, **kw):
        raise NotImplementedError("UavSystem has no collision pass; see ref_nanoflann.cpp")


def collide_snapshot(xyz, arm, prop, mass, crash_mode, rebounce, engine="port", n_threads=1, cap=None):
    """Collision pass on a position snapshot.  Returns (pairs(k,2), forces(n,3), crashed(n))."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
    n = len(xyz)
    arm, prop, mass = (np.ascontiguousarray(np.broadcast_to(a, (n,)), dtype=np.float64) for a in (arm, prop, mass))
    cap = cap or max(1024, 64 * n)
    pairs = np.zeros((cap, 2), dtype=np.int32)
    forces = np.zeros((n, 3))
    crashed = np.zeros(n, dtype=np.uint8)
    if engine == "nanoflann":
        R = ref_lib()
        if R is None:
            raise RuntimeError("oracle/_ref/libref_nanoflann.so not built")
        fn = R.ref_nanoflann_collide
    else:
        fn = lib().orc_collide_port
    cnt = fn(n, _p(xyz), _p(arm), _p(prop), _p(mass), int(crash_mode), float(rebounce), _p(forces), _p(crashed), _p(pairs), cap, n_threads)
    assert cnt <= cap, "pair buffer too small"
    return pairs[:cnt].copy(), forces, crashed
