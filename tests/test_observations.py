"""CPU checks of the references tests/test_observations_gpu.py holds the observation and wrapper kernels to: the numpy restatement of
odometry and the quaternion equals the oracle bit for bit, the long-double rangefinder and heading references with their libm bounds
cover the oracle and glibc, and the restatement tells apart the evaluation orders a kernel could slip into."""
import ctypes as C

import numpy as np

from oracle import binding as O
from test_observations_gpu import (af, assert_bits, assert_range, body_velocity, edge_rotations, heading_reference, height_for_range,
                                   quaternion, random_rotations, random_state, range_edge_state, sincos_bound)


def test_numpy_restatement_equals_the_oracle_bit_for_bit():
    n = 400
    st = random_state(7, n)
    orc = O.OracleSwarm([af("x500")], spawn_xyz=st["x"], n=n)
    orc.set_state(**st)
    od = orc.get_odometry()
    assert_bits(od[:, 3:7], quaternion(st["R"]), "quaternion")
    assert_bits(od[:, 7:10], body_velocity(st["R"], st["v"]), "R^T v")
    assert_bits(orc.get_imu()[:, 6:10], quaternion(st["R"]), "IMU quaternion")


def test_edge_rotations_reach_every_branch_and_the_orders_differ():
    """The edge states take the trace branch and each largest-diagonal branch, ties included, and on random states the evaluation
    orders a kernel could slip into (the trace or a row of R^T v as (a + b) + c, q[j] and q[k] swapped) change some bits."""
    R = edge_rotations()
    M = lambda r, c: R[:, 3 * c + r]
    t = M(0, 0) + (M(1, 1) + M(2, 2))
    other = ~(t > 0.0) & ~np.isnan(R).any(axis=1)
    i = np.where(M(1, 1) > M(0, 0), 1, 0)
    i = np.where(M(2, 2) > np.choose(i, [M(0, 0), M(1, 1)]), 2, i)
    assert (t > 0.0).sum() > 5 and {0, 1, 2} <= set(i[other].tolist()) and np.any(t == 0.0)
    assert np.any(other & (M(0, 0) == M(1, 1)) & (i == 0)) and np.any(other & (M(2, 2) == M(1, 1)) & (i == 1))

    st = random_state(8, 2000, edges=False)
    R, v = st["R"], st["v"]
    q = quaternion(R)
    tp = (R[:, 0] + R[:, 4]) + R[:, 8]
    assert np.any(tp != R[:, 0] + (R[:, 4] + R[:, 8]))
    assert np.any(np.sqrt(tp + 1.0) != q[:, 3] * 2.0)
    bv = np.stack([(R[:, 3 * r] * v[:, 0] + R[:, 3 * r + 1] * v[:, 1]) + R[:, 3 * r + 2] * v[:, 2] for r in range(3)], axis=1)
    assert np.any(bv != body_velocity(R, v))
    Q = quaternion(edge_rotations())
    assert np.any(Q[:, [1, 2, 0, 3]] != Q)


def test_rangefinder_reference_covers_the_oracle():
    R, z, want = range_edge_state()
    n = len(R)
    x = np.stack([np.arange(n) * 3.0, np.zeros(n), z], axis=1)
    orc = O.OracleSwarm([af("x500", ground_enabled=True, ground_z=0.0)], spawn_xyz=x, n=n)
    orc.set_state(x=x, R=R)
    got = orc.get_rangefinder()[:, 0]
    exact = ~np.isnan(want)
    assert_bits(got[exact], want[exact], "exact ranges")
    assert height_for_range(40.0) + 0.01 == 40.0 and got[0] == 40.0 and got[1] == 41.0
    ref, bound = assert_range(got, R, z, np.zeros(n), "edge ranges")
    assert np.isinf(bound).any() and np.all(bound[exact & (R[:, 8] == 1.0)] < 4 * np.spacing(40.0))

    m = 3000
    st = random_state(9, m)
    ok = ~np.isnan(st["R"]).any(axis=1)
    gz = np.where(np.arange(m) % 2 == 0, -1.5, 0.7)
    orc = O.OracleSwarm([af("x500", ground_enabled=True, ground_z=-1.5)], spawn_xyz=st["x"], n=m)
    orc.set_state(**st)
    orc.set_ground_z(0.7, np.arange(1, m, 2))
    got = orc.get_rangefinder()[:, 0]
    ref, bound = assert_range(got[ok], st["R"][ok], st["x"][ok, 2], gz[ok], "random ranges")
    assert np.median(bound[np.isfinite(bound)]) < 1e-13


def test_heading_reference_covers_glibc():
    libm = C.CDLL("libm.so.6")
    for f in ("atan2", "cos", "sin"):
        getattr(libm, f).restype = C.c_double
        getattr(libm, f).argtypes = [C.c_double] * (2 if f == "atan2" else 1)
    R = np.vstack([random_rotations(10, 2000), edge_rotations()])
    R = R[np.isfinite(R[:, :2]).all(axis=1)]
    cut = np.array([cm0 for cm0 in ([-1.0, 0.0], [-2.0, -0.0], [-0.5, 0.0], [-1e-300, -0.0])])
    R[:4, :2] = cut
    h, eh = heading_reference(R)
    got = np.array([libm.atan2(r[1], r[0]) for r in R])
    assert np.all(np.abs(got.astype(np.longdouble) - h) <= eh)
    assert_bits(got[:4], [np.pi, -np.pi, np.pi, -np.pi], "atan2 cut")
    c, s, ec, es = sincos_bound(h, eh)
    assert np.all(np.abs(np.array([libm.cos(x) for x in got]).astype(np.longdouble) - c) <= ec)
    assert np.all(np.abs(np.array([libm.sin(x) for x in got]).astype(np.longdouble) - s) <= es)
