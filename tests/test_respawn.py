"""Episode reset (respawn) without a GPU.  The reference's reset is `uav = UavSystem(params, pos, heading)` (US:144-153);
`RespawnOracle` below does exactly that with the CPU oracle's existing constructor and setters, and is the reference side of the
GPU tests (tests/test_respawn_gpu.py).  Here: its respawn equals a freshly constructed swarm with the same parameters and gains,
bit for bit, and the C++ episode loop through the façade compiles and fails loudly without a device.

`dirty`, `commands`, `fresh_like` and `observe` drive a RespawnOracle, an OracleSwarm and a UavBatch alike."""
import os

import numpy as np
import pytest

from mrs_multirotor_simulator_b200.airframes import airframe
from oracle import binding as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT = 0.01
FF_KINDS = ("acceleration_hdg_rate", "acceleration_hdg", "velocity_hdg", "velocity_hdg_rate")  # oracle kinds 0..3
GAINS = {"mixer": [0.0], "rate": [5.0, 0.05, 0.01], "attitude": [7.0, 0.06, 0.02, 9.0, 1.5], "velocity": [2.5, 0.06, 0.02, 4.5],
         "position": [1.8, 0.12, 0.15, 5.0]}


class RespawnOracle:
    """n independent oracle UavSystems in which respawn(xyz, heading, idx) replaces UAV i by a NEWLY CONSTRUCTED oracle UavSystem
    (its own OracleSwarm of the respawned UAVs): the UAV's current parameters (get_params) with the take-off patch flag it was
    created or last set_params'd with, at the new pose, then the controller gains it was given since its parameters were last
    reset (set_mass / set_ground_z / set_params go through setParams: default gains) applied again.  Everything else forwards
    to the swarm that holds each UAV; the UAVs stay independent, as in the reference (no collision pass here)."""

    def __init__(self, types, type_of_uav=None, spawn_xyz=None, spawn_heading=None, n=None):
        first = O.OracleSwarm(types, type_of_uav=type_of_uav, spawn_xyz=spawn_xyz, spawn_heading=spawn_heading, n=n)
        self.n = first.n
        self.groups = [first]
        self.grp = np.zeros(self.n, dtype=np.int64)
        self.loc = np.arange(self.n, dtype=np.int32)
        tou = np.zeros(self.n, dtype=np.int64) if type_of_uav is None else np.asarray(type_of_uav)
        self.takeoff0 = np.array([first.types[t].takeoff_patch_enabled for t in tou], dtype=np.int32)
        self.gains = [{} for _ in range(self.n)]

    def _each(self, idx, fn):
        idx = np.arange(self.n) if idx is None else np.asarray(idx, dtype=np.int64).reshape(-1)
        g = self.grp[idx]
        for k in np.unique(g):
            sel = np.flatnonzero(g == k)
            fn(self.groups[k], self.loc[idx[sel]], sel)

    @staticmethod
    def _rows(a, n, sel):
        return None if a is None else np.asarray(a, dtype=np.float64).reshape(n, -1)[sel]

    def _n(self, idx):
        return self.n if idx is None else len(idx)

    def set_input(self, mode, payload=None, idx=None):
        n = self._n(idx)
        self._each(idx, lambda s, li, sel: s.set_input(mode, self._rows(payload, n, sel), idx=li))

    def set_feedforward(self, kind, payload, idx=None):
        n = self._n(idx)
        self._each(idx, lambda s, li, sel: s.set_feedforward(kind, self._rows(payload, n, sel), idx=li))

    def apply_force(self, f, idx=None):
        n = self._n(idx)
        self._each(idx, lambda s, li, sel: s.apply_force(self._rows(f, n, sel), idx=li))

    def set_external_moment(self, m, idx=None):
        n = self._n(idx)
        self._each(idx, lambda s, li, sel: s.set_external_moment(self._rows(m, n, sel), idx=li))

    def crash(self, idx=None):
        self._each(idx, lambda s, li, sel: s.crash(idx=li))

    def timeout_input(self, idx=None):
        self._each(idx, lambda s, li, sel: s.timeout_input(idx=li))

    def _params_reset(self, idx):
        for i in (range(self.n) if idx is None else idx):
            self.gains[int(i)] = {}

    def set_mass(self, mass, idx=None):
        m = np.broadcast_to(np.asarray(mass, dtype=np.float64), (self._n(idx),))
        self._each(idx, lambda s, li, sel: s.set_mass(m[sel], idx=li))
        self._params_reset(idx)

    def set_ground_z(self, z, idx=None):
        zz = np.broadcast_to(np.asarray(z, dtype=np.float64), (self._n(idx),))
        self._each(idx, lambda s, li, sel: s.set_ground_z(zz[sel], idx=li))
        self._params_reset(idx)

    def set_params(self, params, idx=None):
        p = params if isinstance(params, O.OrcModelParams) else O.params_from_dict(params)
        self._each(idx, lambda s, li, sel: s.set_params(p, idx=li))
        self._params_reset(idx)
        self.takeoff0[np.arange(self.n) if idx is None else np.asarray(idx)] = p.takeoff_patch_enabled

    def set_controller_params(self, which, values, idx=None):
        self._each(idx, lambda s, li, sel: s.set_controller_params(which, values, idx=li))
        for i in (range(self.n) if idx is None else idx):
            self.gains[int(i)][which] = np.array(values, dtype=np.float64)

    def make_step(self, dt, n_steps=1, n_threads=1):
        for k in np.unique(self.grp):
            self.groups[k].make_step(dt, n_steps, n_threads)

    def get_state(self, idx=None):
        n = self._n(idx)
        out = {k: np.empty((n, w)) for k, w in (("x", 3), ("v", 3), ("R", 9), ("omega", 3), ("motor_rpm", 8), ("v_prev", 3), ("imu", 3))}

        def put(s, li, sel):
            st = s.get_state(li)
            for k in out:
                out[k][sel] = st[k]

        self._each(idx, put)
        return out

    def _gather(self, name, idx, shape, dtype):
        out = np.empty((self._n(idx),) + shape, dtype=dtype)

        def put(s, li, sel):
            out[sel] = getattr(s, name)(li)

        self._each(idx, put)
        return out

    def has_crashed(self, idx=None):
        return self._gather("has_crashed", idx, (), np.int32)

    def get_force(self, idx=None):
        return self._gather("get_force", idx, (3,), np.float64)

    def _one(self, name, uav):
        return getattr(self.groups[self.grp[uav]], name)(int(self.loc[uav]))

    def get_params(self, uav):
        return self._one("get_params", uav)

    def get_pid_state(self, uav=0):
        return self._one("get_pid_state", uav)

    def get_mixer_allocation(self, uav=0):
        return self._one("get_mixer_allocation", uav)

    def respawn(self, xyz, heading, idx=None):
        idx = np.arange(self.n) if idx is None else np.asarray(idx, dtype=np.int64).reshape(-1)
        m = len(idx)
        if m == 0:
            return
        params = []
        for i in idx:
            p = self.get_params(int(i))
            p.takeoff_patch_enabled = int(self.takeoff0[i])
            params.append(p)
        fresh = O.OracleSwarm(params, type_of_uav=np.arange(m, dtype=np.int32), spawn_xyz=np.asarray(xyz, dtype=np.float64).reshape(m, 3),
                              spawn_heading=np.broadcast_to(np.asarray(heading, dtype=np.float64), (m,)), n=m)
        for k, i in enumerate(idx):
            for which, v in self.gains[int(i)].items():
                fresh.set_controller_params(which, v, idx=[k])
        self.groups.append(fresh)
        self.grp[idx] = len(self.groups) - 1
        self.loc[idx] = np.arange(m, dtype=np.int32)


ORACLES = (O.OracleSwarm, RespawnOracle)


def types():
    """x500 / f550 / naki on a ground plane with the take-off patch: UAVs spawned at z = 0 consume it when they lift off."""
    return [airframe(f, ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=True) for f in ("x500", "f550", "naki")]


def type_of(n):
    return (np.arange(n) % 3).astype(np.int32)


def spawn(n, seed=1, z=0.0):
    i = np.arange(n)
    xyz = np.stack([4.0 * (i % 64) + O.u01(seed, 0, i), 4.0 * (i // 64) + O.u01(seed, 1, i), np.full(n, z)], axis=1)
    return xyz, 2.0 * np.pi * O.u01(seed, 2, i) - np.pi


def commands(sw, n, seed, xyz=None):
    """A command of every mode family, by UAV index (mode = 1 + i % 10); returns the modes."""
    i = np.arange(n)
    modes = 1 + i % 10
    u = O.u01(seed, 10, i)
    for mode in range(1, 11):
        k = (i[modes == mode]).astype(np.int32)
        if not len(k):
            continue
        a = u[k]
        if mode == O.ACTUATOR_CMD:
            pl = np.tile(0.55 + 0.1 * a[:, None], (1, 8))
        elif mode == O.CONTROL_GROUP_CMD:
            pl = np.stack([0.02 * a, -0.02 * a, 0.01 * a, 0.6 + 0.05 * a], axis=1)
        elif mode == O.ATTITUDE_RATE_CMD:
            pl = np.stack([0.1 * a, -0.05 * a, 0.2 * a, 0.6 + 0.05 * a], axis=1)
        elif mode == O.ATTITUDE_CMD:
            c, s = np.cos(0.3 * a), np.sin(0.3 * a)
            z0 = np.zeros_like(a)
            pl = np.stack([c, s, z0, -s, c, z0, z0, z0, z0 + 1.0, 0.6 + 0.05 * a], axis=1)
        elif mode == O.TILT_HDG_RATE_CMD:
            pl = np.stack([0.05 * a, -0.05 * a, np.ones_like(a), 0.2 * a, 0.6 + 0.05 * a], axis=1)
        elif mode == O.POSITION_CMD:
            base = xyz[k] if xyz is not None else np.zeros((len(k), 3))
            pl = np.stack([base[:, 0] + 1.0 + a, base[:, 1] - a, base[:, 2] + 2.0 + a, 0.5 * a], axis=1)
        else:  # velocity / acceleration, heading or heading rate
            pl = np.stack([0.5 * a - 0.2, 0.3 - 0.4 * a, 0.8 + 0.3 * a, 0.2 * a], axis=1)
        sw.set_input(mode, pl, idx=k)
    return modes


def _ff(sw, kind, pl, idx):
    sw.set_feedforward(FF_KINDS.index(kind) if isinstance(sw, ORACLES) else kind, pl, idx=idx)


def edits(sw, n):
    """Parameter edits and custom gains that a respawn keeps: set_mass on every 5th UAV, then custom gains on every 4th."""
    m = np.arange(0, n, 5, dtype=np.int32)
    if len(m):
        sw.set_mass(np.array([1.1 * [2.0, 2.3, 7.5][i % 3] for i in m]), idx=m)
    g = np.arange(1, n, 4, dtype=np.int32)
    for which, v in GAINS.items():
        sw.set_controller_params(which, v, idx=g)


def step(sw, n_steps):
    if isinstance(sw, ORACLES):
        sw.make_step(DT, n_steps)
    else:
        for _ in range(n_steps):
            sw.make_step(DT, 1)


def dirty(sw, n, xyz):
    """Everything a respawn has to undo: commands in every mode, feed-forwards, a take-off consumed on the ground, crashes, an
    external force and moment, custom gains, set_mass."""
    edits(sw, n)
    commands(sw, n, 3, xyz)
    f = np.arange(0, n, 3, dtype=np.int32)
    for j, kind in enumerate(FF_KINDS):
        _ff(sw, kind, np.tile([0.1 * (j + 1), -0.05, 0.02, 0.03], (len(f), 1)), f)
    step(sw, 100)
    c = np.arange(2, n, 7, dtype=np.int32)
    sw.crash(idx=c)
    fo = np.arange(1, n, 6, dtype=np.int32)
    sw.apply_force(np.tile([0.4, -0.3, 1.0], (len(fo), 1)), idx=fo)
    mo = np.arange(3, n, 8, dtype=np.int32)
    sw.set_external_moment(np.tile([0.01, -0.02, 0.005], (len(mo), 1)), idx=mo)
    step(sw, 50)


def fresh_like(cls, n, xyz, hdg, **kw):
    """A newly created swarm at the respawn poses with the same parameter edits and gains as a dirtied one."""
    sw = cls(types(), type_of_uav=type_of(n), spawn_xyz=xyz, spawn_heading=hdg, n=n, **kw)
    edits(sw, n)
    return sw


def observe(sw, n):
    st = sw.get_state() if isinstance(sw, ORACLES) else sw.get_full_state()
    st = {k: st[k] for k in ("x", "v", "R", "omega", "motor_rpm", "v_prev", "imu")}
    st["crashed"] = sw.has_crashed()
    st["force"] = sw.get_force()
    st["takeoff"] = np.array([sw.get_params(i).takeoff_patch_enabled for i in range(n)])
    st["mass"] = np.array([sw.get_params(i).mass for i in range(n)])
    return st


def assert_same(a, b, what=""):
    bad = [k for k in a if not np.array_equal(a[k], b[k])]
    assert not bad, f"{what}: {bad} differ"


def test_respawned_oracle_equals_a_fresh_uav_system(oracle_built):
    n = 45
    xyz0, hdg0 = spawn(n, 1)
    a = RespawnOracle(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    dirty(a, n, xyz0)
    before = observe(a, n)
    assert before["crashed"].sum() > 0 and before["takeoff"].sum() < n  # crashed UAVs, and take-offs consumed on the ground
    xyz, hdg = spawn(n, 2)
    xyz[::2, 2] = 0.0  # half of them back on the ground: the take-off patch engages again
    xyz[1::2, 2] = 5.0
    a.respawn(xyz, hdg)
    b = fresh_like(O.OracleSwarm, n, xyz, hdg)
    assert_same(observe(a, n), observe(b, n), "right after the respawn")
    for u in range(n):
        assert np.array_equal(a.get_pid_state(u), b.get_pid_state(u))
        assert np.array_equal(a.get_mixer_allocation(u), b.get_mixer_allocation(u))
    assert observe(a, n)["takeoff"].all()
    for sw in (a, b):
        commands(sw, n, 5, xyz)
    for t in range(10):  # 10 s
        step(a, 100)
        step(b, 100)
        assert_same(observe(a, n), observe(b, n), f"after {t + 1} s")
    for u in range(0, n, 4):
        assert np.array_equal(a.get_pid_state(u), b.get_pid_state(u))


def test_respawned_oracle_subset_leaves_the_others_alone(oracle_built):
    n = 20
    xyz0, hdg0 = spawn(n, 1)
    a = RespawnOracle(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    c = O.OracleSwarm(types(), type_of_uav=type_of(n), spawn_xyz=xyz0, spawn_heading=hdg0, n=n)
    for sw in (a, c):
        dirty(sw, n, xyz0)
    sub = np.array([2, 5, 9, 16], dtype=np.int32)
    a.respawn(xyz0[sub] + 1.0, hdg0[sub], idx=sub)
    for sw in (a, c):
        step(sw, 200)
    rest = np.setdiff1d(np.arange(n), sub)
    oa, oc = observe(a, n), observe(c, n)
    assert_same({k: v[rest] for k, v in oa.items()}, {k: v[rest] for k, v in oc.items()}, "UAVs not respawned")
    assert not oa["crashed"][sub].any()
    assert np.allclose(oa["motor_rpm"][sub, 0], np.array([1170.0, 1360.0, 956.0])[sub % 3], rtol=1e-9)  # no command since: motors at min RPM


def test_episode_loop_compiles_links_and_fails_loudly_without_gpu(tmp_path):
    import subprocess

    import torch
    from test_cpp_facade import build

    exe = build(tmp_path, os.path.join(ROOT, "tests", "cpp", "episode_loop.cpp"))
    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by the gpu test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 3 and "no CUDA device" in r.stderr
