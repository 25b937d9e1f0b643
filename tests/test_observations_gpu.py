"""The rows a learner or a ROS node reads — odometry, IMU, rangefinder, mrsb_pack_observations_device (observe_kernel) — and the rows
the ROS wrapper writes — input-timeout hover synthesis (timeout_input_kernel) and the tracker command (tracker_cmd_kernel) — held
to references of the same arithmetic rather than to a flight tolerance:

* bit for bit wherever the arithmetic is + - * / and sqrt (io_kernels.cu is built with -fmad=false): against the oracle from
  identical states, and against a numpy restatement in the kernel's evaluation order (Eigen's, DESIGN §2) on the GPU's own state
  bits, which also covers states the oracle cannot be given (a padded bucketed batch after flight, sharded handles);
* within a bound derived from CUDA's documented maximum errors where a row goes through acos / cos (the rangefinder) or atan2 /
  sincos (the heading of a timed-out command), against a long-double reference computed from the same float64 inputs.

The CPU checks of these references themselves are in tests/test_observations.py."""
import numpy as np
import pytest

from helpers import rand
from oracle import binding as O

pytestmark = pytest.mark.gpu

U = 2.0 ** -53                              # unit roundoff of float64
EPS_L = float(np.finfo(np.longdouble).eps)  # of the long-double references
# Maximum error of acos, cos, atan2 and sincos in double precision on the device, in ulp of the exact result (CUDA C++ Programming
# Guide, "Mathematical Functions", double-precision table: 2 ulp each).  glibc's are below 1 ulp, so the bounds hold for the oracle.
LIBM_ULP = 2.0

HAD_INPUT = 256                    # FLAG_HAD_INPUT (internal.h)
FF_FLAGS = 16 | 32 | 64 | 128      # FLAG_FF_VEL_HDG_RATE | FLAG_FF_VEL_HDG | FLAG_FF_ACC_HDG_RATE | FLAG_FF_ACC_HDG
CMD0, FF0, SNAP_ROWS = 50, 62, 88  # snapshot record rows: cmd 50-61 (row 60 = cos, 61 = sin of the heading), ff 62-74
ALL_MODES = [O.ACTUATOR_CMD, O.CONTROL_GROUP_CMD, O.ATTITUDE_RATE_CMD, O.ATTITUDE_CMD, O.TILT_HDG_RATE_CMD, O.ACCELERATION_HDG_RATE_CMD,
             O.ACCELERATION_HDG_CMD, O.VELOCITY_HDG_RATE_CMD, O.VELOCITY_HDG_CMD, O.POSITION_CMD]
STRIDE = {O.ACTUATOR_CMD: 8, O.ATTITUDE_CMD: 10, O.TILT_HDG_RATE_CMD: 5}


def af(name, **kw):
    from mrs_multirotor_simulator_b200 import airframe

    return airframe(name, **kw)


# ---- references -------------------------------------------------------------------------------------------------------------------
def quaternion(R):
    """Eigen::Quaterniond(Matrix3d) (x y z w) of column-major rows R [n][9], in float64, in the kernel's and Eigen's order: the trace
    as m00 + (m11 + m22), the branch t > 0, else the largest diagonal entry by strict >."""
    R = np.asarray(R, dtype=np.float64)
    n, a = len(R), np.arange(len(R))

    def M(r, c):
        return R[a, 3 * np.asarray(c) + np.asarray(r)]

    out = np.empty((n, 4))
    with np.errstate(all="ignore"):
        t = M(0, 0) + (M(1, 1) + M(2, 2))
        s = np.sqrt(t + 1.0)
        h = 0.5 / s
        trace = np.stack([(M(2, 1) - M(1, 2)) * h, (M(0, 2) - M(2, 0)) * h, (M(1, 0) - M(0, 1)) * h, 0.5 * s], axis=1)
        i = np.where(M(1, 1) > M(0, 0), 1, 0)
        i = np.where(M(2, 2) > M(i, i), 2, i)
        j = (i + 1) % 3
        k = (j + 1) % 3
        s = np.sqrt(M(i, i) - M(j, j) - M(k, k) + 1.0)
        h = 0.5 / s
        out[a, i] = 0.5 * s
        out[:, 3] = (M(k, j) - M(j, k)) * h
        out[a, j] = (M(j, i) + M(i, j)) * h
        out[a, k] = (M(k, i) + M(i, k)) * h
    return np.where((t > 0.0)[:, None], trace, out)


def body_velocity(R, v):
    """R^T v with each component as Eigen's 3-term product sum: a0 + (a1 + a2)."""
    return np.stack([R[:, 3 * r] * v[:, 0] + (R[:, 3 * r + 1] * v[:, 1] + R[:, 3 * r + 2] * v[:, 2]) for r in range(3)], axis=1)


def odometry(st):
    return np.hstack([st["x"], quaternion(st["R"]), body_velocity(st["R"], st["v"]), st["omega"]])


def imu(st):
    return np.hstack([st["omega"], st["imu"], quaternion(st["R"])])


def range_reference(R, z, ground_z):
    """publishRangefinder (ROSW:401-420) in long double from the float64 inputs, before the clamp, and the largest distance the
    device's result may have from it.  Returns (reference, bound, inverted); inverted rows (bz <= 0 or NaN) read exactly 41.

    The operand of acos, c = bz, is exact in float64 on both sides.  The device's tilt = acos(c) is within 2 ulp(T) of T = acos(c),
    and its cos(tilt) within 2 ulp of cos(tilt), so |cos~ - c| <= sin T * 2 ulp(T) + 2 ulp(|c| + that): relative to c this is
    rho ~ 2^-51 (1 + T tan T), which grows without bound at grazing tilt.  z - ground_z and the division round once each
    (delta = (1 + u)^2 / (1 - rho) - 1 on the quotient q) and the + 0.01 once (u |range|).  The long-double reference carries the
    same terms at its own epsilon."""
    R = np.asarray(R, dtype=np.float64)
    L = np.longdouble
    with np.errstate(all="ignore"):
        c = (-R[:, 6]) * 0.0 + ((-R[:, 7]) * 0.0 + (-R[:, 8]) * -1.0)  # the kernel's acos operand, exact
        T = np.arccos(c.astype(L))
        q = (np.asarray(z, dtype=np.float64).astype(L) - np.asarray(ground_z, dtype=np.float64).astype(L)) / np.cos(T)
        ref = q + L(0.01)  # the float64 literal 0.01 of both sides
        Tf = T.astype(np.float64)
        e_c = np.sin(Tf) * LIBM_ULP * np.spacing(np.abs(Tf))
        e_c = e_c + LIBM_ULP * np.spacing(np.abs(c) + e_c)
        rho = e_c / np.abs(c)
        delta = np.where(rho < 0.5, (1.0 + U) ** 2 / (1.0 - rho) - 1.0, np.inf)
        qa = np.abs(q.astype(np.float64))
        dq = np.where(qa == 0.0, 0.0, qa * delta)  # a zero quotient is exact whatever the divisor (cos of a double is never 0)
        own = 8.0 * EPS_L * (qa * (2.0 + Tf * np.abs(np.tan(Tf))) + np.abs(ref.astype(np.float64)))
        bound = 1.01 * (dq + U * (np.abs(ref.astype(np.float64)) + dq)) + own
    return ref, bound, ~(R[:, 8] > 0.0)


def assert_range(got, R, z, ground_z, what):
    """got within range_reference's bound, or 41 where the clamp may apply (the reference's interval reaches above 40), or exactly
    41 for inverted rows."""
    got = np.asarray(got, dtype=np.float64).reshape(-1)
    ref, bound, inverted = range_reference(R, z, ground_z)
    with np.errstate(invalid="ignore"):
        near = np.abs(got.astype(np.longdouble) - ref) <= bound
        ok = np.where(inverted, got == 41.0, (near & (got <= 40.0)) | ((got == 41.0) & (ref + bound > 40.0)))
        ok |= ~inverted & np.isnan(ref) & np.isnan(got)  # bz > 1 (a raw R): acos gives NaN, and NaN > 40 is false
    bad = np.flatnonzero(~ok)
    assert not len(bad), f"{what}: {len(bad)} ranges outside the bound, e.g. UAV {bad[:4].tolist()}: got {got[bad[:4]].tolist()}, " \
                         f"reference {ref[bad[:4]].astype(float).tolist()} +- {bound[bad[:4]].tolist()}"
    return ref, bound


def heading_reference(R):
    """AttitudeConverter(R).getHeading() = atan2(R10, R00) in long double from the float64 inputs, and the device's bound: 2 ulp."""
    R = np.asarray(R, dtype=np.float64)
    h = np.arctan2(R[:, 1].astype(np.longdouble), R[:, 0].astype(np.longdouble))
    hf = np.abs(h.astype(np.float64))
    return h, LIBM_ULP * np.spacing(hf) + 4.0 * EPS_L * hf


def sincos_bound(h, eh):
    """Bound on the device's cos and sin of its heading against cos and sin of the reference heading h: the heading's own error eh
    (|d sin / dh| <= 1) plus 2 ulp of the result."""
    c, s = np.cos(h), np.sin(h)
    return c, s, eh + LIBM_ULP * np.spacing(np.abs(c.astype(np.float64))) + 4 * EPS_L, eh + LIBM_ULP * np.spacing(np.abs(s.astype(np.float64))) + 4 * EPS_L


def assert_bits(got, want, what):
    """Equal bit for bit (signed zeros included), NaN where the other has NaN (payloads may differ between CPU and GPU)."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    gn, wn = np.isnan(got), np.isnan(want)
    bad = (gn != wn) | (~gn & (got.view(np.uint64) != want.view(np.uint64)))
    where = np.argwhere(bad)[:4].tolist()
    assert not bad.any(), f"{what}: {int(bad.sum())} entries differ, first at {where}: got {got[bad][:4].tolist()}, want {want[bad][:4].tolist()}"


# ---- states -----------------------------------------------------------------------------------------------------------------------
def cm(rows):
    """row-major 3x3 -> 9 column-major doubles"""
    return np.asarray(rows, dtype=np.float64).T.reshape(9)


def axis_angle(axis, angle):
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    K = np.array([[0.0, -a[2], a[1]], [a[2], 0.0, -a[0]], [-a[1], a[0], 0.0]])
    return cm(np.eye(3) + np.sin(angle) * K + (1.0 - np.cos(angle)) * (K @ K))


def edge_rotations():
    """Every branch of Eigen's matrix -> quaternion conversion and its edges."""
    out = [
        cm([[0, 0, 1], [1, 0, 0], [0, 1, 0]]),      # 120 deg about (1,1,1): trace exactly 0, diagonal all 0 -> i = 0
        cm([[0, 1, 0], [0, 0, 1], [1, 0, 0]]),      # 240 deg
        np.eye(3).reshape(9),                       # t = 3
        cm([[1, 0, 0], [0, -1, 0], [0, 0, -1]]),    # 180 deg about x: i = 0
        cm([[-1, 0, 0], [0, 1, 0], [0, 0, -1]]),    # about y: i = 1
        cm([[-1, 0, 0], [0, -1, 0], [0, 0, 1]]),    # about z: i = 2
        cm([[0, 1, 0], [1, 0, 0], [0, 0, -1]]),     # about (1,1,0): m11 == m00 > m22, stays i = 0
        cm([[0, 0, 1], [0, -1, 0], [1, 0, 0]]),     # about (1,0,1): m22 == m00 > m11, stays i = 0
        cm([[-1, 0, 0], [0, 0, 1], [0, 1, 0]]),     # about (0,1,1): m22 == m11 > m00, stays i = 1
        cm([[0, 0, 1], [0, 1, 0], [-1, 0, 0]]),     # 90 deg about y: t = 1
        cm([[1, 0, 0], [0, 0, -1], [0, 1, 0]]),     # 90 deg about x: bz = 0
    ]
    for axis in ([1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 0], [1, 2, 3], [-3, 1, 2], [1, 1, 1]):
        for d in (0.0, 2.0 ** -51, 3 * 2.0 ** -51, 2.0 ** -40):  # within a few ulps of 180 deg, from both sides
            out += [axis_angle(axis, np.pi - d), axis_angle(axis, np.nextafter(np.pi, 4.0) + d)]
    for d in (0.0, 1e-16, -1e-16, 1e-12):  # trace within an ulp or so of 0 in floating point
        out.append(axis_angle([1, 1, 1], 2 * np.pi / 3 + d))
        out.append(axis_angle([1, -2, 0.5], 2 * np.pi / 3 + d))
    # raw, non-orthonormal matrices are allowed by setState (MM:424-433)
    k = np.arange(6)
    raw = np.stack([rand(61, s, 6, -2, 2) for s in range(9)], axis=1)
    raw[k % 2 == 0] *= 1e-3
    out += list(raw)
    out.append(cm([[-1, 0.5, 0], [0.5, -1, 0], [0, 0, -1]]))  # trace -3, ties
    out.append(cm([[2, 0, 0], [0, 2, 0], [0, 0, 2]]))
    out.append(np.zeros(9))
    # NaN entries: on the diagonal, off it, in bz
    for pos in (0, 4, 8, 5, 1, 6):
        r = np.eye(3).reshape(9).copy()
        r[pos] = np.nan
        out.append(r)
    return np.array(out)


def random_rotations(seed, n):
    q = np.stack([rand(seed, s, n, -1, 1) for s in range(4)], axis=1)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    x, y, z, w = q.T
    rows = [[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
            [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
            [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]]
    return np.stack([rows[r][c] for c in range(3) for r in range(3)], axis=1)  # column-major


def random_state(seed, n, z=(-5.0, 45.0), edges=True):
    """x, v, R, omega for n UAVs: random rotations, with edge_rotations() on the last UAVs (so they straddle a tile boundary)."""
    R = random_rotations(seed, n)
    if edges:
        E = edge_rotations()
        m = min(n, len(E))
        R[n - m:] = E[:m]
    return dict(x=np.stack([rand(seed, 10, n, -50, 50), rand(seed, 11, n, -50, 50), rand(seed, 12, n, *z)], axis=1),
                v=np.stack([rand(seed, 13 + c, n, -5, 5) for c in range(3)], axis=1), R=R,
                omega=np.stack([rand(seed, 16 + c, n, -3, 3) for c in range(3)], axis=1))


def height_for_range(target):
    """A z with fl(z + 0.01) == target exactly (upright UAV over ground 0: the range is z / cos(acos(1)) + 0.01 = z + 0.01)."""
    z = target - 0.01
    while z + 0.01 > target:
        z = np.nextafter(z, -np.inf)
    while z + 0.01 < target:
        z = np.nextafter(z, np.inf)
    assert z + 0.01 == target
    return z


def range_edge_state():
    """Upright, inverted, grazing and below-ground UAVs: rows (R, z) and what each must read over a ground plane at 0.
    The last element is the exact expected range where one exists (NaN: judged by the bound alone)."""
    I = np.eye(3).reshape(9)
    lying = cm([[1, 0, 0], [0, 0, -1], [0, 1, 0]])
    rows = []

    def bz(value):
        r = lying.copy() if value <= 0 else I.copy()
        r[8] = value
        return r

    for z in (height_for_range(40.0), height_for_range(np.nextafter(40.0, 41.0)), 3.25, -2.5, 0.0, 39.99, 40.5):
        rows.append((I, z, 41.0 if z + 0.01 > 40.0 else z + 0.01))  # acos(1) = 0 and cos(0) = 1 exactly
    for v in (0.0, -0.0):  # lying or inverted: bz = +-0 is not > 0
        for z in (0.0, 5.0, -5.0):
            rows.append((bz(v), z, 41.0))
    for z, want in ((0.0, 0.01), (5.0, np.nan), (-5.0, np.nan)):  # smallest subnormal bz: the branch is taken; 0 / cos~ + 0.01 = 0.01
        rows.append((bz(5e-324), z, want))
    for v in (1e-300, 1e-12, 1e-8, 1e-3, 0.05, 0.5, 0.999999):  # towards grazing tilt
        r = axis_angle([1, 2, 0], np.arccos(v))
        for z in (0.0, 0.004, 1.0, 39.0):
            rows.append((r, z, np.nan))
    rows.append((cm([[1, 0, 0], [0, -1, 0], [0, 0, -1]]), 5.0, 41.0))  # upside down
    R = np.array([r[0] for r in rows])
    return R, np.array([r[1] for r in rows]), np.array([r[2] for r in rows])


# ---- handles ----------------------------------------------------------------------------------------------------------------------
TYPES3 = (("x500", -1.5), ("naki", 0.5), ("f550", 0.0))


def three_types():
    return [af(name, ground_enabled=True, ground_z=gz) for name, gz in TYPES3]


def bucketed(n=3 * 1000 + 7, z=(-5.0, 45.0), seed=3):
    """3 airframes interleaved (each bucket ends in a partial tile), every UAV in a random state"""
    from mrs_multirotor_simulator_b200 import UavBatch

    tou = (np.arange(n) % 3).astype(np.int32)
    st = random_state(seed, n, z)
    gpu = UavBatch(three_types(), type_of_uav=tou, spawn_xyz=st["x"], n=n)
    assert gpu.device_view().slot_of_uav  # bucketed: slots are permuted
    gpu.set_state(**st)
    return gpu, tou


def ground_of(tou):
    return np.array([gz for _, gz in TYPES3])[tou]


def snapshot_image(gpu):
    """(rows [88][n], flags [n], modes [n]) of a snapshot's host image: a 48-byte header, then the rows, flags and input modes."""
    snap = gpu.snapshot()
    snap.save()
    b = snap.to_bytes()
    snap.free()
    n = gpu.n
    assert len(b) == 48 + 709 * n
    return (np.frombuffer(b, np.float64, SNAP_ROWS * n, 48).reshape(SNAP_ROWS, n).copy(), np.frombuffer(b, np.uint32, n, 48 + 704 * n).copy(),
            np.frombuffer(b, np.uint8, n, 48 + 708 * n).copy())


def packed(gpu, stride, sentinel=-123.25):
    import torch

    buf = torch.full((gpu.n, stride), sentinel, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    gpu.pack_observations_device(buf.data_ptr(), stride)
    gpu.sync()
    out = buf.cpu().numpy()
    assert np.all(out[:, 17:] == sentinel), "columns past the 17 packed ones were written"
    return out[:, :17]


def index_lists(n, tou):
    """permuted; crossing tiles and buckets; holding the last UAV; empty"""
    rng = np.random.default_rng(n)
    return [rng.permutation(n)[: max(1, n // 3)], np.concatenate([np.arange(120, min(n, 140)), np.flatnonzero(tou == 2)[-5:], [0]]),
            np.array([n - 1, 0, n - 1]), np.array([], dtype=np.int32)]


def make_shards(types, tou, spawn, cuts):
    from mrs_multirotor_simulator_b200 import UavBatch

    n = len(spawn)
    out = []
    for b, e in zip(cuts[:-1], cuts[1:]):
        out.append(UavBatch(types, type_of_uav=tou, spawn_xyz=spawn[b:e], n=e - b, n_global=n, shard_begin=b))
    return out


# ---- identical states: the GPU equals the oracle bit for bit ---------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 127, 128, 129, 300])
def test_identical_states_equal_the_oracle_bit_for_bit(n):
    """x, the quaternion, R^T v and omega of get_odometry and get_imu equal the oracle's bit for bit from the same set_state; so does
    the numpy restatement.  The rangefinder is within the libm bound of the long-double reference on both."""
    from mrs_multirotor_simulator_b200 import UavBatch

    st = random_state(7, n)
    types = [af("x500", ground_enabled=True, ground_z=-1.5)]
    orc = O.OracleSwarm(types, spawn_xyz=st["x"], n=n)
    gpu = UavBatch(types, spawn_xyz=st["x"], n=n)
    for s in (orc, gpu):
        s.set_state(**st)
    od_o, od_g = orc.get_odometry(), gpu.get_odometry()
    assert_bits(od_g, od_o, "odometry, GPU vs oracle")
    assert_bits(od_g, odometry(gpu.get_full_state()), "odometry, GPU vs numpy")
    im_o, im_g = orc.get_imu(), gpu.get_imu()
    assert_bits(im_g[:, [0, 1, 2, 6, 7, 8, 9]], im_o[:, [0, 1, 2, 6, 7, 8, 9]], "IMU angular velocity and orientation, GPU vs oracle")
    assert_bits(im_g, imu(gpu.get_full_state()), "IMU, GPU vs numpy")
    gz = np.full(n, -1.5)
    ok = ~np.isnan(st["R"]).any(axis=1)
    for what, rg in (("GPU", gpu.get_rangefinder()), ("oracle", orc.get_rangefinder())):
        assert_range(rg[ok], st["R"][ok], st["x"][ok, 2], gz[ok], f"rangefinder, {what}")
    assert_bits(gpu.get_rangefinder()[~ok], orc.get_rangefinder()[~ok], "ranges of NaN attitudes, GPU vs oracle")


def test_rangefinder_edges_exact_and_bounded():
    """Clamp at exactly 40.0 and its successor, bz = +0 / -0 / the smallest subnormal, below ground, grazing tilt: exact where the
    range is exact, within the libm bound elsewhere, equal to the oracle where both are exact."""
    from mrs_multirotor_simulator_b200 import UavBatch

    R, z, want = range_edge_state()
    n = len(R)
    x = np.stack([np.arange(n) * 3.0, np.zeros(n), z], axis=1)
    types = [af("x500", ground_enabled=True, ground_z=0.0)]
    orc = O.OracleSwarm(types, spawn_xyz=x, n=n)
    gpu = UavBatch(types, spawn_xyz=x, n=n)
    for s in (orc, gpu):
        s.set_state(x=x, R=R)
    rg, ro = gpu.get_rangefinder()[:, 0], orc.get_rangefinder()[:, 0]
    exact = ~np.isnan(want)
    assert_bits(rg[exact], want[exact], "exact ranges, GPU")
    assert_bits(ro[exact], want[exact], "exact ranges, oracle")
    assert rg[0] == 40.0 and rg[1] == 41.0 and rg[3] < 0.0
    assert_range(rg, R, z, np.zeros(n), "rangefinder edges, GPU")
    assert_range(ro, R, z, np.zeros(n), "rangefinder edges, oracle")
    pk = packed(gpu, 24)
    assert_bits(pk[:, 16], rg, "packed range")


# ---- the GPU's own bits: bucketed, padded, uniform, index-addressed, packed ------------------------------------------------------
@pytest.mark.parametrize("layout", ["bucketed-3x1000+7", "uniform-58001"])
def test_rows_equal_the_numpy_restatement_after_flight(layout):
    """After flight, get_odometry / get_imu (for every index list) and pack_observations_device (strides 17 and 24, columns 17-23
    untouched) equal the numpy restatement on get_full_state bit for bit; ranges are within the libm bound."""
    from mrs_multirotor_simulator_b200 import UavBatch

    if layout.startswith("bucketed"):
        gpu, tou = bucketed(z=(2.0, 30.0))
        n = gpu.n
    else:
        n = 58001
        st = random_state(5, n, z=(2.0, 30.0))
        tou = np.zeros(n, dtype=np.int32)
        gpu = UavBatch([af("x500", ground_enabled=True, ground_z=-1.5)], spawn_xyz=st["x"], n=n)
        gpu.set_state(**st)
    cmd = np.stack([rand(9, 1, n, -3, 3), rand(9, 2, n, -3, 3), rand(9, 3, n, -1, 1), rand(9, 4, n, -1, 1)], axis=1)
    gpu.set_input(O.VELOCITY_HDG_RATE_CMD, cmd)
    for _ in range(5):
        gpu.make_step(0.01, 10)
    st = gpu.get_full_state()
    od, im = odometry(st), imu(st)
    assert_bits(gpu.get_odometry(), od, f"{layout}: odometry")
    assert_bits(gpu.get_imu(), im, f"{layout}: IMU")
    rg = gpu.get_rangefinder()
    gz = ground_of(tou) if layout.startswith("bucketed") else np.full(n, -1.5)
    assert_range(rg, st["R"], st["x"][:, 2], gz, f"{layout}: rangefinder")
    assert len(np.unique(rg)) > n // 3 and np.any(rg == 41.0) and np.any(rg < 40.0)
    for idx in index_lists(n, tou):
        assert_bits(gpu.get_odometry(idx), od[idx], f"{layout}: odometry of {len(idx)} listed UAVs")
        assert_bits(gpu.get_imu(idx), im[idx], f"{layout}: IMU of {len(idx)} listed UAVs")
        assert_bits(gpu.get_rangefinder(idx), rg[idx], f"{layout}: range of {len(idx)} listed UAVs")
    want = np.hstack([od, st["imu"], rg])
    for stride in (17, 24):
        assert_bits(packed(gpu, stride), want, f"{layout}: packed observations, stride {stride}")


def test_ground_z_subset_of_a_bucketed_batch_before_any_step_and_after_set_mass():
    """set_ground_z on a subset that crosses buckets, read before any step (the parameter table is uploaded by the read itself), and
    again after set_mass on the same UAVs: upright UAVs read exactly z - ground_z + 0.01 of their own ground plane, like the oracle."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 3 * 1000 + 7
    tou = (np.arange(n) % 3).astype(np.int32)
    x = np.stack([rand(12, 0, n, -50, 50), rand(12, 1, n, -50, 50), rand(12, 2, n, -3, 42)], axis=1)
    orc = O.OracleSwarm(three_types(), type_of_uav=tou, spawn_xyz=x, n=n)
    gpu = UavBatch(three_types(), type_of_uav=tou, spawn_xyz=x, n=n)
    sub = np.concatenate([np.arange(1, n, 7), [n - 1]])
    gz = np.round(rand(12, 3, len(sub), -2, 3), 3)
    gz_all = ground_of(tou)
    gz_all[sub] = gz
    want = np.where(x[:, 2] - gz_all + 0.01 > 40.0, 41.0, x[:, 2] - gz_all + 0.01)
    for s in (orc, gpu):
        s.set_ground_z(gz, sub)
    for when in ("before any step", "after set_mass"):
        rg = gpu.get_rangefinder()[:, 0]
        assert_bits(rg, want, f"ranges {when}")
        assert_bits(rg, orc.get_rangefinder()[:, 0], f"ranges {when}, GPU vs oracle")
        assert_bits(packed(gpu, 17)[:, 16], want, f"packed ranges {when}")
        for s in (orc, gpu):
            s.set_mass(rand(12, 4, len(sub), 1.0, 3.0), sub)


# ---- sharded handles -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cuts", [(0, 1000, 3007), (0, 700, 1901, 3007)])
def test_sharded_observations_equal_unsharded(cuts):
    """Shards cut inside tiles and buckets: concatenated, their odometry, IMU, ranges and packed rows equal the unsharded handle's
    bit for bit, with per-UAV ground planes set on a subset that spans the cuts."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = cuts[-1]
    tou = (np.arange(n) % 3).astype(np.int32)
    st = random_state(21, n, z=(0.0, 30.0))
    st["R"][::4] = np.eye(3).reshape(9)  # upright: the range is exact, so a wrong ground plane is visible
    whole = UavBatch(three_types(), type_of_uav=tou, spawn_xyz=st["x"], n=n)
    shards = make_shards(three_types(), tou, st["x"], cuts)
    sub = np.arange(cuts[1] - 40, cuts[1] + 45)
    gz = rand(22, 0, len(sub), -3, 3)
    whole.set_state(**st)
    whole.set_ground_z(gz, sub)
    for sh in shards:
        b, e = sh.shard_begin, sh.shard_begin + sh.n
        sh.set_state(**{k: v[b:e] for k, v in st.items()})
        mine = (sub >= b) & (sub < e)
        if mine.any():
            sh.set_ground_z(gz[mine], sub[mine] - b)
    for name, get in (("odometry", lambda s: s.get_odometry()), ("IMU", lambda s: s.get_imu()), ("range", lambda s: s.get_rangefinder()),
                      ("packed", lambda s: packed(s, 24))):
        assert_bits(np.concatenate([get(sh) for sh in shards]), get(whole), f"{name}, shards {cuts} vs unsharded")
    gz_all = ground_of(tou)
    gz_all[sub] = gz
    up = np.arange(0, n, 4)
    rg = whole.get_rangefinder()[up, 0]
    want = st["x"][up, 2] - gz_all[up] + 0.01
    assert_bits(rg, np.where(want > 40.0, 41.0, want), "upright ranges over each UAV's own ground plane")


# ---- outputs switched off ---------------------------------------------------------------------------------------------------------
def test_imu_switched_off_is_a_state_error():
    import torch

    from mrs_multirotor_simulator_b200._lib import MrsbError

    gpu, _ = bucketed(n=300)
    od, rg = gpu.get_odometry(), gpu.get_rangefinder()
    gpu.set_outputs(imu=False)
    buf = torch.zeros((gpu.n, 17), dtype=torch.float64, device="cuda")
    for call in (gpu.get_imu, gpu.get_imu_acceleration, lambda: gpu.pack_observations_device(buf.data_ptr(), 17)):
        with pytest.raises(MrsbError) as e:
            call()
        assert e.value.code == -5  # MRSB_ERR_STATE
    assert_bits(gpu.get_odometry(), od, "odometry with the IMU off")
    assert_bits(gpu.get_rangefinder(), rg, "range with the IMU off")
    gpu.set_outputs(imu=True)
    gpu.get_imu()


# ---- IMU acceleration after one step ----------------------------------------------------------------------------------------------
# Measured on one NVIDIA B200 (1000 W power limit): the largest |GPU - oracle| of the IMU acceleration after one step from these
# identical states is 5.33e-15 m/s^2 without FLAG_VPREV (|a| up to 12 m/s^2) and 2.28e-13 m/s^2 with it (|a| up to 660 m/s^2: the
# step from the stored v_prev to v is seen as one jump).  The tolerance is five times the measured gap.
IMU_ONE_STEP_TOL = {False: 5 * 5.33e-15, True: 5 * 2.28e-13}


@pytest.mark.parametrize("vprev", [False, True])
def test_imu_acceleration_after_one_step(vprev):
    """One step from identical states (set_state with v: v_prev holds the old v, FLAG_VPREV; without v: v_prev reads as v)."""
    from mrs_multirotor_simulator_b200 import UavBatch

    n = 300
    st = random_state(31, n, edges=False)
    st["R"] = np.tile(np.eye(3).reshape(9), (n, 1))
    st["R"][::2] = axis_angle([1, 2, 0.3], 0.4)
    st["omega"] *= 0.1
    if not vprev:
        del st["v"]
    rpm = np.stack([rand(31, 40 + m, n, 3000, 5000) for m in range(4)] + [np.zeros(n)] * 4, axis=1)
    types = [af("x500")]
    orc = O.OracleSwarm(types, spawn_xyz=st["x"], n=n)
    gpu = UavBatch(types, spawn_xyz=st["x"], n=n)
    cmd = np.stack([rand(31, 50 + m, n, 0.4, 0.7) for m in range(8)], axis=1)
    for s in (orc, gpu):
        s.set_state(motor_rpm=rpm, **st)
        s.set_input(O.ACTUATOR_CMD, cmd)
        s.make_step(0.01)
    a_o, a_g = orc.get_imu()[:, 3:6], gpu.get_imu()[:, 3:6]
    gap = float(np.max(np.abs(a_o - a_g)))
    print(f"IMU acceleration after one step, vprev={vprev}: max |GPU - oracle| = {gap:.3e}, max |a| = {np.max(np.abs(a_o)):.3e}")
    assert np.max(np.abs(a_o)) > 1.0
    assert gap <= IMU_ONE_STEP_TOL[vprev], gap
    assert_bits(a_g, gpu.get_imu_acceleration(), "get_imu == get_imu_acceleration")


# ---- timeout_input ----------------------------------------------------------------------------------------------------------------
def test_timeout_input_every_mode_on_a_bucketed_batch():
    """Every mode on the padded bucketed batch, an index list across buckets: copied and constant command rows exact, the heading and
    its cos / sin within the libm bound (exactly +-pi on the atan2 cut), FLAG_HAD_INPUT cleared on the listed UAVs only, modes kept,
    nothing else of any UAV changed."""
    gpu, tou = bucketed()
    n = gpu.n
    modes = np.array(ALL_MODES + [O.INPUT_UNKNOWN])[(np.arange(n) * 7) % 11]
    HDG = [O.POSITION_CMD, O.VELOCITY_HDG_CMD, O.ACCELERATION_HDG_CMD]
    R = gpu.get_full_state()["R"]
    # R10 = +-0 with R00 < 0, where atan2 gives exactly +-pi
    cut = np.concatenate([np.flatnonzero(np.isin(modes, HDG))[::37][:20], np.flatnonzero(modes == O.ATTITUDE_CMD)[::61][:6]])
    R[cut] = np.array([cm([[-1.0 - j % 3, 0.0, 0.0], [0.0 if j % 2 else -0.0, -1.0, 0.0], [0.0, 0.0, 1.0]]) for j in range(len(cut))])
    gpu.set_state(R=R)
    for m in ALL_MODES:
        idx = np.flatnonzero(modes == m)
        w = STRIDE.get(m, 4)
        gpu.set_input(m, np.stack([rand(40 + m, c, len(idx), -3, 3) for c in range(w)], axis=1), idx)
    rows_a, flags_a, modes_a = snapshot_image(gpu)
    assert np.array_equal(modes_a, modes)
    listed = np.random.default_rng(5).permutation(n)[: 2 * n // 3]
    listed = np.unique(np.concatenate([listed, cut, [n - 1]]))[::-1].copy()
    gpu.timeout_input(listed)
    rows_b, flags_b, modes_b = snapshot_image(gpu)

    on = np.zeros(n, dtype=bool)
    on[listed] = True
    assert np.array_equal(modes_b, modes_a)
    assert np.array_equal(flags_b, np.where(on, flags_a & ~np.uint32(HAD_INPUT), flags_a))
    assert np.any(flags_a[on] & HAD_INPUT) and not np.any(flags_b[on] & HAD_INPUT)

    want = rows_a.copy()
    libm = np.zeros_like(want, dtype=bool)
    C = lambda r: CMD0 + r
    x = rows_a[0:3]
    for m in ALL_MODES:
        sel = on & (modes == m)
        if m == O.POSITION_CMD:
            want[C(0):C(3), sel] = x[:, sel]
        if m in (O.VELOCITY_HDG_CMD, O.ACCELERATION_HDG_CMD):
            want[C(0):C(3), sel] = 0.0
        if m in (O.POSITION_CMD, O.VELOCITY_HDG_CMD, O.ACCELERATION_HDG_CMD):
            libm[[C(3), C(10), C(11)]] |= sel
        if m in (O.VELOCITY_HDG_RATE_CMD, O.ACCELERATION_HDG_RATE_CMD, O.ATTITUDE_RATE_CMD, O.CONTROL_GROUP_CMD):
            want[C(0):C(4), sel] = 0.0
        if m == O.ATTITUDE_CMD:
            for r, v in ((2, 0.0), (5, 0.0), (6, 0.0), (7, 0.0), (8, 1.0), (9, 0.0)):
                want[C(r), sel] = v
            libm[[C(0), C(1), C(3), C(4)]] |= sel
        if m == O.TILT_HDG_RATE_CMD:
            want[C(0):C(5), sel] = np.array([0.0, 0.0, 1.0, 0.0, 0.0])[:, None]
        if m == O.ACTUATOR_CMD:
            want[C(0):C(8), sel] = 0.0
    assert_bits(np.where(libm, 0.0, rows_b), np.where(libm, 0.0, want), "copied, constant and untouched snapshot rows")

    h, eh = heading_reference(R)
    ch, sh, ec, es = sincos_bound(h, eh)
    L = np.longdouble
    finite = np.isfinite(R[:, :2]).all(axis=1)  # NaN in R00 or R10: a NaN heading
    hdg = on & np.isin(modes, HDG)
    att = on & (modes == O.ATTITUDE_CMD)
    assert (hdg & finite).sum() > 300 and (att & finite).sum() > 100 and (hdg & ~finite).any()
    assert np.all(np.isnan(rows_b[[C(3), C(10), C(11)]][:, hdg & ~finite])) and np.all(np.isnan(rows_b[[C(0), C(1)]][:, att & ~finite]))
    hdg &= finite
    att &= finite
    for what, got, ref, bound, sel in (("heading", rows_b[C(3)], h, eh, hdg), ("cos", rows_b[C(10)], ch, ec, hdg), ("sin", rows_b[C(11)], sh, es, hdg),
                                       ("attitude cos", rows_b[C(0)], ch, ec, att), ("attitude sin", rows_b[C(1)], sh, es, att)):
        err = np.abs(got[sel].astype(L) - ref[sel])
        bad = np.flatnonzero(~(err <= bound[sel]))
        assert not len(bad), f"{what}: {len(bad)} outside the libm bound, e.g. got {got[sel][bad[:3]].tolist()}, reference {ref[sel][bad[:3]].astype(float).tolist()}"
    assert_bits(rows_b[C(3), att], -rows_b[C(1), att], "attitude: R01 = -sin")
    assert_bits(rows_b[C(4), att], rows_b[C(0), att], "attitude: R11 = cos")
    on_cut = cut[hdg[cut]]
    assert len(on_cut) >= 10
    assert_bits(rows_b[C(3), on_cut], np.copysign(np.pi, R[on_cut, 1]), "heading on the atan2 cut")
    assert np.any(np.signbit(R[on_cut, 1])) and not np.all(np.signbit(R[on_cut, 1]))


# ---- set_tracker_cmd with an index list -------------------------------------------------------------------------------------------
def test_tracker_cmd_with_an_index_list_on_a_bucketed_batch():
    """Feed-forward rows 62-74 and the four feed-forward flag bits of the listed UAVs equal a numpy model of callbackTrackerCmd
    (ROSW:987-1022) exactly; nothing of the other UAVs changes."""
    gpu, tou = bucketed()
    n = gpu.n
    early = np.arange(3, n, 5)
    gpu.set_feedforward("velocity_hdg_rate", np.stack([rand(50, c, len(early), -1, 1) for c in range(4)], axis=1), early)
    gpu.set_feedforward("acceleration_hdg", np.stack([rand(51, c, len(early), -1, 1) for c in range(4)], axis=1), early)
    listed = np.random.default_rng(9).permutation(n)[: n // 2]
    listed = np.concatenate([listed[listed != n - 1], [n - 1]])
    k = len(listed)
    use = np.stack([(np.arange(k) >> b) % 2 for b in range(4)], axis=1).astype(float)
    use[use == 1] = np.array([1.0, -2.5, np.nan, 1e-300])[np.arange(int((use == 1).sum())) % 4]  # any non-zero means "use"
    use[(use == 0) & (np.arange(k)[:, None] % 3 == 0)] = -0.0                                       # -0.0 == 0: do not
    rows = np.hstack([np.stack([rand(52, c, k, -2, 2) for c in range(7)], axis=1), use])
    rows[::11, 0] = -0.0
    rows_a, flags_a, modes_a = snapshot_image(gpu)
    gpu.set_tracker_cmd(rows, listed)
    rows_b, flags_b, modes_b = snapshot_image(gpu)

    uh, uv, ur, ua = (rows[:, 7 + c] != 0.0 for c in range(4))
    v = np.stack([np.where(uh, rows[:, 0], 0.0), np.where(uh, rows[:, 1], 0.0), np.where(uv, rows[:, 2], 0.0)])
    a = np.where(ua, rows[:, 3:6].T, 0.0)
    want = rows_a.copy()
    want[FF0:FF0 + 13, listed] = np.vstack([v, v, a, a, np.where(ur, rows[:, 6], 0.0)[None]])
    assert_bits(rows_b, want, "snapshot rows after set_tracker_cmd")
    want_flags = flags_a.copy()
    want_flags[listed] |= FF_FLAGS
    assert np.array_equal(flags_b, want_flags) and np.array_equal(modes_b, modes_a)
    assert uh.any() and (~uh).any() and ur.any() and (~ur).any()
