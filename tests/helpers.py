"""Shared helpers for the parity tests: build the SAME swarm in the CPU oracle and in libmrsb,
drive both with the same seeded commands, compare state within the stated tolerances.

Tolerances (DESIGN.md §5; SURVEY §8c): after 10 s of simulated flight
    |dx| <= 1e-9 m, |dv| <= 1e-9 m/s, |dR| <= 1e-10, |domega| <= 1e-8 rad/s, |drpm| <= 1e-6 RPM.
"""
import ctypes as C
import hashlib
import json
import os

import numpy as np

from oracle import binding as O

TOL = {"x": 1e-9, "v": 1e-9, "R": 1e-10, "omega": 1e-8, "motor_rpm": 1e-6, "v_prev": 1e-9, "imu": 1e-6}


def digest(*values):
    """8 hex digits of the SHA-256 of the exact bytes of `values` (arrays, dicts of arrays, ctypes structures, scalars):
    a stored digest pins a computed value bit for bit."""
    h = hashlib.sha256()
    for v in values:
        if isinstance(v, dict):
            h.update(digest(*(v[k] for k in sorted(v))).encode())
        elif isinstance(v, C.Structure):
            h.update(bytes(v))
        else:
            h.update(np.ascontiguousarray(v, dtype=np.asarray(v).dtype).tobytes())
    return h.hexdigest()[:8]


class StoredResults:
    """The reference side of a test module, with or without the reference's own build (oracle/_ref/libref_uavsystem.so).

    With the build, the tests run against it (mode "live"), or store the digest of every observation they make of it
    (states, PID states, crash flags, forces, mixer rows, parameters), in order and per test, in `path` (mode "record":
    MRSB_RECORD_REFERENCE=1).  Without it, the restatement stands in and each of its observations must equal the stored
    digest (mode "check"): the same comparisons, against the stored results."""

    def __init__(self, path):
        built = O.refsys_lib() is not None
        self.path = path
        self.mode = ("record" if os.environ.get("MRSB_RECORD_REFERENCE") else "live") if built else "check"
        self.base = O.RefSwarm if built else O.OracleSwarm
        self.stored, self.test, self.seen = None, None, ""

    def observe(self, value):
        if self.mode == "live":
            return value
        d = digest(value)
        if self.mode == "check":
            i = len(self.seen)
            assert self.stored["tests"].get(self.test, "")[i:i + 8] == d, \
                f"{self.test}: observation {i // 8} of the reference side differs from the stored result"
        self.seen += d
        return value

    def swarm(self):
        """The reference side's swarm class."""
        log = self

        class Observed(self.base):
            def get_state(self, idx=None):
                return log.observe(super().get_state(idx))

            def get_pid_state(self, uav=0):
                return log.observe(super().get_pid_state(uav))

            def has_crashed(self, idx=None):
                return log.observe(super().has_crashed(idx))

            def get_force(self, idx=None):
                return log.observe(super().get_force(idx))

            def get_mixer_allocation(self, uav=0):
                return log.observe(super().get_mixer_allocation(uav))

            def get_params(self, uav):
                return log.observe(super().get_params(uav))

        return Observed

    def module(self):
        """Body of a module-scoped fixture: loads the stored digests, or writes them after recording."""
        if self.mode == "record":
            self.stored = {"source": "the reference's own UavSystem sources (oracle/_ref/libref_uavsystem.so)", "tests": {}}
        elif self.mode == "check":
            with open(self.path) as f:
                self.stored = json.load(f)
        yield
        if self.mode == "record":
            with open(self.path, "w") as f:
                json.dump(self.stored, f, indent=0, sort_keys=True)

    def run(self, test):
        """Body of a per-test fixture."""
        self.test, self.seen = test, ""
        yield
        if self.mode == "record" and self.seen:
            self.stored["tests"][test] = self.seen
        elif self.mode == "check":
            assert self.seen == self.stored["tests"].get(test, ""), f"{test}: fewer observations of the reference side than stored"


def grid_spawn(n, pitch=4.0, z=0.0):
    side = int(np.ceil(np.sqrt(n)))
    i = np.arange(n)
    return np.stack([pitch * (i % side), pitch * (i // side), np.full(n, z)], axis=1).astype(np.float64)


def rand(seed, stream, n, lo, hi):
    return lo + (hi - lo) * O.u01(seed, stream, np.arange(n))


def make_pair(types, type_of_uav, spawn_xyz, spawn_heading=None, device=0):
    from mrs_multirotor_simulator_b200 import UavBatch

    n = len(spawn_xyz)
    if spawn_heading is None:
        spawn_heading = np.zeros(n)
    orc = O.OracleSwarm(types, type_of_uav=type_of_uav, spawn_xyz=spawn_xyz, spawn_heading=spawn_heading, n=n)
    gpu = UavBatch(types, type_of_uav=type_of_uav, spawn_xyz=spawn_xyz, spawn_heading=spawn_heading, n=n, device=device)
    return orc, gpu


def max_diffs(orc, gpu, fields=("x", "v", "R", "omega", "motor_rpm", "v_prev", "imu")):
    so = orc.get_state()
    sg = gpu.get_full_state()
    return {k: float(np.max(np.abs(so[k] - sg[k]))) if so[k].size else 0.0 for k in fields}


def assert_parity(orc, gpu, tol=None, scale=1.0, what=""):
    tol = tol or TOL
    so = orc.get_state()
    sg = gpu.get_full_state()
    bad = []
    for k, t in tol.items():
        assert np.all(np.isfinite(so[k])), f"oracle {k} not finite {what}"
        d = float(np.max(np.abs(so[k] - sg[k]))) if so[k].size else 0.0
        if not d <= t * scale:
            bad.append(f"{k}: {d:.3e} > {t * scale:.1e}")
    assert not bad, f"parity {what}: " + "; ".join(bad)
