"""The collision pass against the reference at the edges of its predicates and settings.

Every comparison here is with the reference's own collision loop on the GPU's own positions (pairs and crash flags from
ENGINE, forces from the port, which sums in the same ascending-j order as the kernels), or with the oracle's flight:

  A  contact thresholds that are not symmetric in floating point (SIM:342), and nanoflann's strict search ball d2 < 3.0
     (NF:305-309) for an airframe whose contact distance is above 3.0, on every pass kind: the full pass, the rebuild pass of a
     neighbour-list handle, a list-only pass, the crowded path and a shard cut;
  B  exactly 8 and exactly 9 list candidates (MRSB_NL_CAP = 8);
  C  set_params / set_mass: the per-UAV geometry table the pass reads must follow every edit;
  D  rebounce values other than 100, changed between passes, through single calls and the tick graph;
  E  crash mode without collisions enabled (SIM:299-301);
  F  more pairs than the pair buffer holds.

Positions near the origin make every coordinate difference exact, so that nf_dist2 takes exactly the value aimed at.
"""
import ctypes as C

import numpy as np
import pytest

from helpers import assert_parity, make_pair, rand
from oracle import binding as O
from test_collisions_gpu import ENGINE, af, geometry, sorted_pairs
from test_neighbour_lists_gpu import batch
from test_sharded_gpu import exchange, make_shards

pytestmark = pytest.mark.gpu

MRSB_ERR_CAPACITY = -4  # include/mrsb.h


def nf_dist2(p, q):
    """nanoflann's L2 for dim 3 (NF:479-484) in Python doubles: ((d0*d0) + d1*d1) + d2*d2, no contraction."""
    d0, d1, d2 = float(p[0]) - float(q[0]), float(p[1]) - float(q[1]), float(p[2]) - float(q[2])
    return (d0 * d0 + d1 * d1) + d2 * d2


def crit(a, b):
    """SIM:342: ((arm_i + prop_i) + arm_j) + prop_j"""
    return ((a["arm_length"] + a["prop_radius"]) + b["arm_length"]) + b["prop_radius"]


def offset_at(target):
    """(dx, dy, 0) with nf_dist2((0,0,0), (dx,dy,0)) == target exactly: a nextafter search around dy = sqrt(target - dx^2)."""
    for dx in (0.5, 0.6, 0.7, 0.4, 0.3, 0.8):
        dy = float(np.sqrt(target - dx * dx))
        for direction in (np.inf, -np.inf):
            v = dy
            for _ in range(64):
                if nf_dist2((0.0, 0.0, 0.0), (dx, v, 0.0)) == target:
                    return np.array([dx, v, 0.0])
                v = float(np.nextafter(v, direction))
    raise AssertionError(f"no exact offset for {target!r}")


def below(v):
    return float(np.nextafter(v, -np.inf))


def above(v):
    return float(np.nextafter(v, np.inf))


def ring(centre, axis, r, k=9):
    """k points on a circle of radius r around `centre`, in the plane normal to `axis`"""
    a = np.asarray(axis, dtype=np.float64) / np.linalg.norm(axis)
    u = np.cross(a, [0.0, 0.0, 1.0] if abs(a[2]) < 0.9 else [1.0, 0.0, 0.0])
    u /= np.linalg.norm(u)
    v = np.cross(a, u)
    t = 2.0 * np.pi * np.arange(k) / k
    return centre + r * (np.cos(t)[:, None] * u + np.sin(t)[:, None] * v)


def place(pairs, fillers=0, filler_type=0):
    """pairs: [(type_a, type_b, offset)], one pair per z level 12 m apart, a at (0, 0, z) and b at (0, 0, z) + offset.  Member a of
    pair k is UAV k and member b UAV m + k (m pairs): every pair straddles the index m.  `fillers`: that many UAVs of
    `filler_type` on a ring of radius 2.2 m around each pair's axis (2.25..2.4 m from both members: list candidates outside the
    search ball).  Returns tou, xyz and the [(a, b)] indices."""
    m = len(pairs)
    xyz = np.zeros((2 * m, 3))
    tou = np.zeros(2 * m, dtype=np.int32)
    extra, extra_t = [], []
    for k, (ta, tb, off) in enumerate(pairs):
        z = 5.0 + 12.0 * k
        xyz[k] = (0.0, 0.0, z)
        xyz[m + k] = np.array([0.0, 0.0, z]) + off
        tou[k], tou[m + k] = ta, tb
        if fillers:
            extra.append(ring(0.5 * (xyz[k] + xyz[m + k]), off, 2.2, fillers))
            extra_t += [filler_type] * fillers
    if extra:
        xyz = np.concatenate([xyz] + extra)
        tou = np.concatenate([tou, np.array(extra_t, dtype=np.int32)])
    assert all(nf_dist2(xyz[k], xyz[m + k]) == nf_dist2((0, 0, 0), pairs[k][2]) for k in range(m))  # the differences are exact
    return tou, xyz, [(k, m + k) for k in range(m)]


def candidates(xyz, r):
    """per UAV, the number of other UAVs with nf_dist2 < r^2, after checking that no distance is within 0.1 m of r"""
    d = np.sqrt(((xyz[:, None, :] - xyz[None, :, :]) ** 2).sum(-1))
    off = ~np.eye(len(xyz), dtype=bool)
    assert not np.any(off & (np.abs(d - r) < 0.1)), "a distance too close to the list radius"
    return ((d < r) & off).sum(1)


def reference(types, tou, xyz, crash, rebounce, geom=None):
    arm, prop, mass = geom if geom is not None else geometry(types, tou)
    cap = max(1024, len(xyz) * len(xyz) if len(xyz) <= 600 else 64 * len(xyz))
    pairs, _, crashed = O.collide_snapshot(xyz, arm, prop, mass, crash, rebounce, engine=ENGINE, n_threads=8, cap=cap)
    _, forces, _ = O.collide_snapshot(xyz, arm, prop, mass, crash, rebounce, engine="port", n_threads=8, cap=cap)
    return sorted_pairs(pairs), forces, crashed.astype(np.int32)


def assert_pass(b, ref, what):
    pairs, forces, crashed = ref
    assert np.array_equal(pairs, b.get_collision_pairs()), what
    assert np.array_equal(forces, b.get_force()), what
    assert np.array_equal(crashed, b.has_crashed()), what


def pass_kinds(types, tou, xyz, crash, rebounce):
    """Every kind of pass on the same positions: (kind, handle) after the full pass of a handle without lists, the rebuild pass
    of a list handle and a list-only pass of that handle (a stepping launch that moves nobody: without iterate_without_input, UAVs
    that never had an input are not stepped)."""
    full = batch(types, tou, xyz, lists=False)
    lists = batch(types, tou, xyz, lists=True)
    for b in (full, lists):
        b.set_iterate_without_input(False)
        b.set_collisions(True, crash, rebounce)
        b.set_pair_capacity(4096)
    full.handle_collisions()
    yield "full pass", full
    lists.handle_collisions()
    info = lists.collision_info()
    assert (info["passes"], info["rebuilds"]) == (1, 1), info
    yield "rebuild pass", lists
    lists.make_step(0.01)
    lists.handle_collisions()
    info = lists.collision_info()
    assert (info["passes"], info["rebuilds"]) == (2, 1), info  # list-only
    assert np.array_equal(lists.get_state()["x"], xyz)
    yield "list-only pass", lists


def asymmetric_pairs():
    """f450-t650 and t650-naki at the one-ulp window between their two directed thresholds, and one double either side."""
    names = ("f450", "t650", "naki")
    types = [af(t) for t in names]
    spec, window = [], []
    for a, b in ((0, 1), (1, 2)):
        lo, hi = sorted((crit(types[a], types[b]), crit(types[b], types[a])))
        assert hi == above(lo)  # one ulp apart: the pair exists in one direction only at d2 == lo
        if crit(types[a], types[b]) < hi:
            a, b = b, a  # a: the UAV whose threshold is the larger one
        window.append(len(spec) + 1)
        spec += [(a, b, offset_at(below(lo))), (a, b, offset_at(lo)), (a, b, offset_at(hi))]
    return types, spec, window


def assert_asymmetric(ref_pairs, ab, spec, window):
    present = {tuple(p) for p in ref_pairs}
    for k, (a, b) in enumerate(ab):
        if k in window:  # (a, b) only
            assert (a, b) in present and (b, a) not in present, spec[k]
        elif k - 1 in window:  # the next double above: neither
            assert (a, b) not in present and (b, a) not in present, spec[k]
        else:  # the next double below: both
            assert (a, b) in present and (b, a) in present, spec[k]


# ---- A: threshold edges --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("crash", [False, True])
def test_asymmetric_contact_thresholds_on_every_pass_kind(crash):
    types, spec, window = asymmetric_pairs()
    tou, xyz, ab = place(spec)
    ref = reference(types, tou, xyz, crash, 100.0)
    assert_asymmetric(ref[0], ab, spec, window)
    if crash:  # the reference marks the neighbour j of (i, j): one of the two UAVs of the one-way pair only
        for k in window:
            a, b = ab[k]
            assert ref[2][b] == 1 and ref[2][a] == 0
    for kind, b in pass_kinds(types, tou, xyz, crash, 100.0):
        assert_pass(b, ref, kind)


def large_airframe_pairs():
    """An airframe with contact distance 3.3 > 3.0 (nanoflann's search ball decides) next to x500 (3.0 > 2.05 with it)."""
    big = af("x500", arm_length=1.2, prop_radius=0.45)
    types = [big, af("x500")]
    assert crit(big, big) > 3.1 and crit(big, types[1]) < below(3.0)
    third = np.array([1.0, 1.0, 1.0])
    assert nf_dist2((0, 0, 0), third) == 3.0
    over = np.array([1.0, 1.45, 0.0])
    assert 3.0 < nf_dist2((0, 0, 0), over) < crit(big, big)
    spec = [(0, 0, third), (0, 0, offset_at(below(3.0))), (0, 0, over), (0, 1, third), (0, 1, offset_at(below(3.0))), (1, 0, offset_at(2.0))]
    return types, spec


@pytest.mark.parametrize("crash", [False, True])
def test_search_ball_of_a_large_airframe_on_every_pass_kind(crash):
    types, spec = large_airframe_pairs()
    tou, xyz, ab = place(spec)
    ref = reference(types, tou, xyz, crash, 100.0)
    present = {tuple(p) for p in ref[0]}
    # within the contact distance but not inside the ball (d2 == 3.0, 3.1): no pair; just inside it: both directions
    for k in (0, 2, 3):
        assert ab[k] not in present and ab[k][::-1] not in present, spec[k]
    assert ab[1] in present and ab[1][::-1] in present
    assert ab[4] not in present and ab[5] in present and ab[5][::-1] in present
    for kind, b in pass_kinds(types, tou, xyz, crash, 100.0):
        assert_pass(b, ref, kind)


@pytest.mark.parametrize("crash", [False, True])
def test_crowded_uavs_at_the_threshold_edges(crash):
    """The UAVs of the edge pairs above with nine x500 between sqrt(3) and 2.9 m of them: more candidates than a list holds, so
    they walk the table (check_crowded) on the rebuild pass and on the list-only pass."""
    big_types, big_spec = large_airframe_pairs()
    asym_types, asym_spec, window = asymmetric_pairs()
    types = big_types + asym_types  # 0 big, 1 x500, 2 f450, 3 t650, 4 naki
    spec = big_spec[:3] + [(a + 2, b + 2, off) for a, b, off in asym_spec]
    tou, xyz, ab = place(spec, fillers=9, filler_type=1)
    m = len(spec)
    cand = candidates(xyz, batch(types, tou, xyz).collision_info()["list_radius"])
    assert np.all(cand[:2 * m] >= 10)  # the pair partner and nine fillers
    ref = reference(types, tou, xyz, crash, 100.0)
    present = {tuple(p) for p in ref[0]}
    assert ab[0] not in present and ab[1] in present and ab[2] not in present
    assert_asymmetric(ref[0], ab[3:], spec[3:], window)
    for kind, b in pass_kinds(types, tou, xyz, crash, 100.0):
        if kind != "full pass":
            assert b.collision_info()["crowded_uavs"] == int(np.sum(cand > 8)), kind
        assert_pass(b, ref, kind)


@pytest.mark.parametrize("crash", [False, True])
def test_asymmetric_pairs_across_a_shard_cut(crash):
    """Two handles on one GPU, the members of every edge pair on different sides of the cut: the owner of each UAV decides its
    own pairs and its own crash flag."""
    types, spec, window = asymmetric_pairs()
    big_types, big_spec = large_airframe_pairs()
    types = types + big_types  # 0 f450, 1 t650, 2 naki, 3 big, 4 x500
    spec = spec + [(a + 3, b + 3, off) for a, b, off in big_spec]
    tou, xyz, ab = place(spec)
    m = len(spec)
    ref = reference(types, tou, xyz, crash, 100.0)
    assert_asymmetric(ref[0], ab[:6], spec[:6], window)
    assert all(a < m <= b for a, b in ab)
    shards = make_shards(types, tou, xyz, (0, m, 2 * m))
    for sh in shards:
        sh.set_collisions(True, crash, 100.0)
        sh.publish_positions()
    exchange(shards)
    for sh in shards:
        sh.handle_collisions_gathered()
    pairs = sorted_pairs(np.concatenate([sh.get_collision_pairs() for sh in shards]))
    assert np.array_equal(ref[0], pairs)
    assert np.array_equal(ref[1], np.concatenate([sh.get_force() for sh in shards]))
    assert np.array_equal(ref[2], np.concatenate([sh.has_crashed() for sh in shards]))


# ---- B: the list-capacity boundary ---------------------------------------------------------------------------------------
def test_eight_and_nine_list_candidates():
    """A cube of x500 with its centre (9 UAVs, 8 candidates each) and one with its centre and a UAV 0.5 m from the centre (10
    UAVs, 9 candidates each): only the second is crowded.  Then 100 ticks of the two clusters drifting, pairs and forces every
    tick."""
    cube = 0.8 * np.array([[x, y, z] for x in (-1, 1) for y in (-1, 1) for z in (-1, 1)], dtype=np.float64)
    a = np.concatenate([cube, [[0.0, 0.0, 0.0]]]) + [0.0, 0.0, 10.0]
    b = np.concatenate([cube, [[0.0, 0.0, 0.0], [0.5, 0.0, 0.0]]]) + [30.0, 0.0, 10.0]
    xyz = np.concatenate([a, b])
    n = len(xyz)
    types = [af("x500")]
    tou = np.zeros(n, dtype=np.int32)
    gpu = batch(types, tou, xyz)
    cand = candidates(xyz, gpu.collision_info()["list_radius"])
    assert sorted(set(cand.tolist())) == [8, 9] and int(np.sum(cand == 8)) == 9 and int(np.sum(cand == 9)) == 10
    gpu.set_collisions(True, False, 10.0)
    gpu.handle_collisions()
    assert gpu.collision_info()["crowded_uavs"] == int(np.sum(cand > 8)) == 10
    assert_pass(gpu, reference(types, tou, xyz, False, 10.0), "first pass")
    gpu.set_input(O.VELOCITY_HDG_RATE_CMD, np.tile([0.6, 0.3, 0.0, 0.0], (n, 1)))
    total = 0
    for tick in range(100):
        gpu.make_step(0.01)
        gpu.handle_collisions()
        ref = reference(types, tou, gpu.get_state()["x"], False, 10.0)
        assert_pass(gpu, ref, f"tick {tick}")
        total += len(ref[0])
    info = gpu.collision_info()
    assert total > 0 and info["rebuilds"] < info["passes"], info


# ---- C: geometry edits against the oracle --------------------------------------------------------------------------------
def crowd(n, pitch, seed):
    side = int(np.ceil(np.sqrt(n)))
    k = np.arange(n)
    return np.stack([pitch * (k % side) + rand(seed, 0, n, -0.3, 0.3), pitch * (k // side) + rand(seed, 1, n, -0.3, 0.3), rand(seed, 2, n, 9.0, 10.0)], axis=1)


# weak enough that UAVs pass through each other: a strong push would move every UAV in contact out of the enlarged contact distance
# before the edit is reverted, and the revert would change no pair
REBOUNCE_C = 4.0


@pytest.mark.parametrize("kind", ["uniform", "bucketed"])
def test_geometry_edits_vs_oracle(kind):
    names = ("x500",) if kind == "uniform" else ("x500", "f550", "naki")
    n = 2025 if kind == "uniform" else 2400
    tou = (np.arange(n) % len(names)).astype(np.int32)
    types = [af(t) for t in names]
    spawn = crowd(n, 1.25, seed=23)
    orc, gpu = make_pair(types, tou, spawn)
    assert gpu.collision_info()["neighbour_lists"]
    cmd = np.stack([rand(9, 1, n, -1, 1), rand(9, 2, n, -1, 1), rand(9, 3, n, -0.2, 0.2), rand(9, 4, n, -0.5, 0.5)], axis=1)
    for s in (orc, gpu):
        s.set_input(O.VELOCITY_HDG_RATE_CMD, cmd)
        s.set_collisions(True, False, REBOUNCE_C)
    gpu.set_pair_capacity(16 * n)
    geom = [g.copy() for g in geometry(types, tou)]

    def tick(step, what):
        if step:
            orc.make_step(0.01, 1, 8)
            gpu.make_step(0.01)
        po = orc.handle_collisions(engine=ENGINE, n_threads=8)
        gpu.handle_collisions()
        assert np.array_equal(sorted_pairs(po), gpu.get_collision_pairs()), what
        assert np.array_equal(orc.has_crashed(), gpu.has_crashed()), what
        _, forces, _ = O.collide_snapshot(gpu.get_state()["x"], *geom, False, REBOUNCE_C, engine="port", n_threads=8)
        assert np.array_equal(forces, gpu.get_force()), what
        return sorted_pairs(po), forces

    def fly(what):
        before = gpu.collision_info()
        last = None
        for t in range(100):
            last = tick(True, f"{what}, tick {t}")
        after = gpu.collision_info()
        assert after["passes"] - before["passes"] > after["rebuilds"] - before["rebuilds"], (what, before, after)  # list-only passes
        return last

    edited = np.arange(0, n, 7)  # every airframe's bucket
    massed = np.arange(3, n, 5)
    pairs, forces = fly("before the edits")
    # set_params with larger arms and propellers: contact distances grow
    for t, name in enumerate(names):
        idx = edited[tou[edited] == t]
        p = af(name, arm_length=1.5 * types[t]["arm_length"], prop_radius=1.4 * types[t]["prop_radius"])
        for s in (orc, gpu):
            s.set_params(p, idx=idx)
        geom[0][idx], geom[1][idx] = p["arm_length"], p["prop_radius"]
    c, _ = tick(False, "set_params, no step")
    assert len(c) > len(pairs)
    pairs, forces = fly("after set_params")
    # set_mass on another subset: only the rebounce weights change
    mass = geom[2][massed] * (1.0 + 0.1 * (1 + massed % 4))
    for s in (orc, gpu):
        s.set_mass(mass, idx=massed)
    geom[2][massed] = mass
    c, f = tick(False, "set_mass, no step")
    assert np.array_equal(c, pairs) and not np.array_equal(f, forces)
    pairs, forces = fly("after set_mass")
    # set_params back to the shipped airframe
    for t, name in enumerate(names):
        idx = edited[tou[edited] == t]
        for s in (orc, gpu):
            s.set_params(types[t], idx=idx)
        geom[0][idx], geom[1][idx], geom[2][idx] = types[t]["arm_length"], types[t]["prop_radius"], types[t]["mass"]
    c, _ = tick(False, "set_params back, no step")
    assert not np.array_equal(c, pairs)
    fly("after set_params back")
    assert_parity(orc, gpu, what=f"{kind} crowd with geometry edits")


# ---- D: rebounce values ---------------------------------------------------------------------------------------------------
def flying_crowd(n, lists, seed=31):
    types = [af("x500"), af("f550")]
    tou = (np.arange(n) % 2).astype(np.int32)
    b = batch(types, tou, crowd(n, 1.3, seed), lists=lists)
    b.set_input(O.VELOCITY_HDG_RATE_CMD, np.stack([rand(seed, 1, n, -1, 1), rand(seed, 2, n, -1, 1), np.zeros(n), rand(seed, 4, n, -0.5, 0.5)], axis=1))
    b.set_pair_capacity(16 * n)
    return types, tou, b


@pytest.mark.parametrize("lists", [True, False])
def test_rebounce_values_through_calls_and_the_tick_graph(lists):
    n = 1024
    types, tou, b = flying_crowd(n, lists)
    pushed = pairs_at_zero = 0
    for rebounce, via in ((37.25, "calls"), (0.0, "calls"), (37.25, "run"), (0.0, "run"), (37.25, "run"), (0.0, "calls"), (37.25, "calls")):
        b.set_collisions(True, False, rebounce)
        for t in range(6):
            if via == "run":
                b.run(0.01, 1)
            else:
                b.make_step(0.01)
                b.handle_collisions()
            ref = reference(types, tou, b.get_state()["x"], False, rebounce)
            assert_pass(b, ref, f"rebounce {rebounce} through {via}, tick {t}")
            if rebounce:
                pushed += int(np.any(ref[1] != 0.0, axis=1).sum())
            else:
                pairs_at_zero += len(ref[0])
    assert pushed > 0 and pairs_at_zero > 0
    if lists:
        info = b.collision_info()
        assert info["rebuilds"] < info["passes"], info


# ---- E: crash mode without collisions enabled ------------------------------------------------------------------------------
@pytest.mark.parametrize("lists", [True, False])
def test_crash_only_pass(lists):
    n = 1024
    types, tou, b = flying_crowd(n, lists, seed=37)
    b.set_collisions(False, True, 100.0)
    b.apply_force(np.ones((n, 3)))
    crashed = np.zeros(n, dtype=np.int32)
    total = 0
    for t in range(40):
        if t < 20:
            b.make_step(0.01)
            b.handle_collisions()
        else:
            b.run(0.01, 1)
        pairs, _, c = reference(types, tou, b.get_state()["x"], True, 100.0)
        crashed |= c
        assert np.array_equal(pairs, b.get_collision_pairs()), t
        assert np.array_equal(crashed, b.has_crashed()), t
        assert not b.get_force().any(), t
        total += len(pairs)
    assert total > 0 and crashed.any()


# ---- F: a full pair buffer --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("crash", [False, True])
def test_full_pair_buffer(crash):
    """Fewer pair slots than pairs: the true count is reported with MRSB_ERR_CAPACITY, forces and crash flags are complete; after
    raising the capacity the next pass returns every pair.  On a rebuild pass and on list-only passes."""
    n = 400
    types = [af("x500"), af("t650")]
    tou = (np.arange(n) % 2).astype(np.int32)
    xyz = crowd(n, 1.0, seed=41)
    ref = reference(types, tou, xyz, crash, 100.0)
    k = len(ref[0]) // 3
    assert k > 50
    b = batch(types, tou, xyz)
    b.set_iterate_without_input(False)
    b.set_collisions(True, crash, 100.0)
    b.set_pair_capacity(k)

    def full_buffer(what, rebuilds):
        cnt = C.c_int64(-1)
        assert b._L.mrsb_get_collision_pairs(b.h, None, 0, C.byref(cnt)) == MRSB_ERR_CAPACITY, what
        assert cnt.value == len(ref[0]), what
        assert np.array_equal(ref[1], b.get_force()), what
        assert np.array_equal(ref[2], b.has_crashed()), what
        assert b.collision_info()["rebuilds"] == rebuilds, what

    b.handle_collisions()
    full_buffer("rebuild pass", 1)
    b.make_step(0.01)  # nobody has had an input: nobody moves
    b.handle_collisions()
    full_buffer("list-only pass", 1)
    b.set_pair_capacity(4 * len(ref[0]))
    b.make_step(0.01)
    b.handle_collisions()
    assert b.collision_info()["rebuilds"] == 1
    assert_pass(b, ref, "list-only pass after raising the capacity")
