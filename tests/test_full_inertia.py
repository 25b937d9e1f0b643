"""A full (non-diagonal) inertia tensor against a plain reference: Euler's equations for a rigid body.

With min_rpm = 0 and ActuatorCmd zeros the motors stay at 0 RPM, so the only torque is the external moment and the body rates
follow Euler's equations alone, w' = J^-1 (tau - w x J w) (MM:346-350), whatever R, x and v do.  The simulator integrates them
with classic RK4 (MM:220-286); integrated with the same RK4, dt and step count in long double, they give the body rates up to
rounding.  This pins the oracle's full-J path (the j_diagonal == 0 branch of the kernels is checked against the same reference in
tests/test_staged_edits_gpu.py).

Tolerance: integrating the same states with the same RK4 in float64 instead of long double moves w by at most 5.6e-13 rad/s after
10 s (generic states, where the intermediate axis amplifies rounding; 1.3e-14 near the major and minor axes).  That gap is what
rounding amplification alone does; OMEGA_TOL allows about five times it (the oracle's gap: 4.9e-13).  Leaving out the off-diagonal
terms of J moves w by 6.9 rad/s.
"""
import numpy as np

from oracle import binding as O

DT, STEPS = 0.01, 1000  # 10 s
OMEGA_TOL = 3e-12  # rad/s; see the module docstring
# World-frame angular momentum R J w with zero moment: plain long-double RK4 of (R, w) at this dt drifts by 1.2e-8 (relative) in
# 10 s, the simulator, which re-orthonormalises R in every RK stage (MM:249-253, 314-316), by 7.5e-8.  Wrong J in either half: O(1).
L_DRIFT_TOL = 2.5e-7


def _rot(a, b, c):
    ca, sa, cb, sb, cc, sc = np.cos(a), np.sin(a), np.cos(b), np.sin(b), np.cos(c), np.sin(c)
    return (np.array([[ca, -sa, 0], [sa, ca, 0], [0, 0, 1]]) @ np.array([[cb, 0, sb], [0, 1, 0], [-sb, 0, cb]])
            @ np.array([[1, 0, 0], [0, cc, -sc], [0, sc, cc]]))


def full_inertia(principal=(0.030, 0.046, 0.066), angles=(0.4, -0.3, 0.25)):
    """Symmetric positive-definite J with off-diagonal terms: principal moments `principal` about the columns of a fixed rotation."""
    Q = _rot(*angles)
    J = Q @ np.diag(principal) @ Q.T
    return 0.5 * (J + J.T)


def free_body_airframe(J):
    """An x500-sized quadrotor whose motors can stand still (min_rpm = 0), without ground or take-off patch: with ActuatorCmd
    zeros its body rates obey Euler's equations alone."""
    return dict(n_motors=4, mass=2.0, arm_length=0.25, body_height=0.1, motor_time_constant=0.03, air_resistance_coeff=0.30, kf=2.7087e-7,
                km=0.07, prop_radius=0.15, min_rpm=0.0, max_rpm=7800.0,
                allocation=[[-0.707, 0.707, 0.707, -0.707], [-0.707, 0.707, -0.707, 0.707], [-1, -1, 1, 1], [1, 1, 1, 1]],
                J=np.asarray(J).tolist(), g=9.81, ground_enabled=False, takeoff_patch_enabled=False)


def euler_states(J, gidx):
    """Seeded initial body rates and external moments of the UAVs `gidx` (global indices): gidx % 3 == 0 near the major axis,
    1 near the minor axis, 2 in a generic direction; 1-4 rad/s; every fourth UAV has zero moment, the others up to 2 mN m."""
    gidx = np.asarray(gidx)
    u = lambda s: O.u01(7, s, gidx)
    d = np.stack([u(0) - 0.5, u(1) - 0.5, u(2) - 0.5], axis=1)
    d /= np.linalg.norm(d, axis=1)[:, None]
    _, axes = np.linalg.eigh(J)  # ascending principal moments: column 0 minor, column 2 major
    cls = gidx % 3
    w0 = np.where(cls[:, None] == 2, d, np.where(cls[:, None] == 0, axes[:, 2], axes[:, 0]) + 0.02 * d)
    w0 = w0 / np.linalg.norm(w0, axis=1)[:, None] * (1.0 + 3.0 * u(3))[:, None]
    tau = np.stack([u(4) - 0.5, u(5) - 0.5, u(6) - 0.5], axis=1) * 0.004
    tau[gidx % 4 == 0] = 0.0
    return w0, tau


def _inv3(a):
    c = np.empty_like(a)
    c[0, 0], c[0, 1], c[0, 2] = a[1, 1] * a[2, 2] - a[1, 2] * a[2, 1], a[0, 2] * a[2, 1] - a[0, 1] * a[2, 2], a[0, 1] * a[1, 2] - a[0, 2] * a[1, 1]
    c[1, 0], c[1, 1], c[1, 2] = a[1, 2] * a[2, 0] - a[1, 0] * a[2, 2], a[0, 0] * a[2, 2] - a[0, 2] * a[2, 0], a[0, 2] * a[1, 0] - a[0, 0] * a[1, 2]
    c[2, 0], c[2, 1], c[2, 2] = a[1, 0] * a[2, 1] - a[1, 1] * a[2, 0], a[0, 1] * a[2, 0] - a[0, 0] * a[2, 1], a[0, 0] * a[1, 1] - a[0, 1] * a[1, 0]
    return c / (a[0, 0] * c[0, 0] + a[0, 1] * c[1, 0] + a[0, 2] * c[2, 0])


def euler_rk4(J, w0, tau, dt=DT, steps=STEPS, dtype=np.longdouble):
    """Classic RK4 of w' = J^-1 (tau - w x J w) for rows of w0 / tau, computed in `dtype`; returns float64."""
    J, w, tau, dt = J.astype(dtype), w0.astype(dtype), tau.astype(dtype), dtype(dt)
    Ji = _inv3(J)

    def f(w):
        Jw = w @ J.T
        return (tau - np.cross(w, Jw)) @ Ji.T

    h = dt / 2
    for _ in range(steps):
        k1 = f(w)
        k2 = f(w + h * k1)
        k3 = f(w + h * k2)
        k4 = f(w + dt * k3)
        w = w + dt / 6 * (k1 + 2 * k2 + 2 * k3 + k4)
    return w.astype(np.float64)


def angular_momentum(state, J):
    """World-frame R J w of each row of a state dict (R stored column-major, 9 doubles)."""
    R = state["R"].reshape(-1, 3, 3).transpose(0, 2, 1)
    return np.einsum("nij,jk,nk->ni", R, J, state["omega"])


def test_oracle_full_inertia_follows_eulers_equations():
    """The oracle's body rates over 10 s against the long-double RK4 of Euler's equations; with zero moment, R J w is conserved."""
    J = full_inertia()
    assert np.all(np.linalg.eigvalsh(J) > 0) and np.min(np.abs(J[~np.eye(3, dtype=bool)])) > 1e-3
    n = 300
    gidx = np.arange(n)
    w0, tau = euler_states(J, gidx)
    ref = euler_rk4(J, w0, tau)
    gap = np.max(np.abs(euler_rk4(J, w0, tau, dtype=np.float64) - ref))
    assert gap <= OMEGA_TOL / 4, f"float64 vs long double gap {gap:.3e}: OMEGA_TOL no longer reflects these states"
    orc = O.OracleSwarm([free_body_airframe(J)], spawn_xyz=np.tile([0.0, 0.0, 100.0], (n, 1)), spawn_heading=O.u01(7, 9, gidx) * 6 - 3, n=n)
    orc.set_state(omega=w0)
    orc.set_external_moment(tau)
    orc.set_input(O.ACTUATOR_CMD, np.zeros((n, 8)))
    L0 = angular_momentum(orc.get_state(), J)
    orc.make_step(DT, STEPS)
    s = orc.get_state()
    assert np.all(s["motor_rpm"] == 0.0)
    d = np.max(np.abs(s["omega"] - ref))
    assert d <= OMEGA_TOL, f"omega differs from Euler's equations by {d:.3e} rad/s"
    # the generic states tumble: not a test of the initial state
    assert np.min(np.max(np.abs(s["omega"] - w0), axis=1)[gidx % 3 == 2]) > 1e-2
    zero = ~tau.any(axis=1)
    L = angular_momentum(s, J)
    drift = np.max(np.linalg.norm(L - L0, axis=1)[zero] / np.linalg.norm(L0, axis=1)[zero])
    assert drift <= L_DRIFT_TOL, f"world-frame angular momentum drifted by {drift:.3e}"
