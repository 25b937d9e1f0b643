"""Neighbour observations (mrsb_pack_neighbours_device): the k nearest UAVs within a radius, for every UAV, on the device.

The reference side is `reference()` below: candidate pairs from a KD-tree with a slack radius, then the library's exact predicate
recomputed in numpy (elementwise IEEE operations, so the same bits as the kernel's nf_dist2), sorted by (i, d2, j).  Every GPU
comparison is bit-exact: indices, counts and rows."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

MAX_K = 16
ERR_INVALID, ERR_STATE = -1, -5


def dist2(a, b):
    """d2 = ((dx*dx) + dy*dy) + dz*dz with dx = b - a, rowwise, one IEEE operation at a time."""
    d = b - a
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def reference(pos, vel, r, k):
    """(idx [n][k], rows [n][6k], count [n]) as include/mrsb.h defines them, vectorised."""
    pos = np.asarray(pos, dtype=np.float64)
    vel = np.asarray(vel, dtype=np.float64)
    n = len(pos)
    ok = np.flatnonzero(np.isfinite(pos).all(axis=1))
    pr = np.zeros((0, 2), dtype=np.int64)
    if len(ok) >= 2:
        pr = ok[cKDTree(pos[ok]).query_pairs(r * (1.0 + 1e-6), output_type="ndarray").reshape(-1, 2)]
    i = np.concatenate([pr[:, 0], pr[:, 1]])
    j = np.concatenate([pr[:, 1], pr[:, 0]])
    d2 = dist2(pos[i], pos[j])
    keep = d2 < r * r
    i, j, d2 = i[keep], j[keep], d2[keep]
    o = np.lexsort((j, d2, i))
    i, j = i[o], j[o]
    count = np.bincount(i, minlength=n).astype(np.int32)
    first = np.concatenate([[0], np.cumsum(count)[:-1]])
    rank = np.arange(len(i)) - first[i]
    sel = rank < k
    i, j, rank = i[sel], j[sel], rank[sel]
    idx = np.full((n, k), -1, dtype=np.int32)
    idx[i, rank] = j
    rows = np.zeros((n, 6 * k))
    for c in range(3):
        rows[i, 6 * rank + c] = pos[j, c] - pos[i, c]
        rows[i, 6 * rank + 3 + c] = vel[j, c] - vel[i, c]
    return idx, rows, count


def brute_force(pos, vel, r, k):
    n = len(pos)
    idx = np.full((n, k), -1, dtype=np.int32)
    rows = np.zeros((n, 6 * k))
    count = np.zeros(n, dtype=np.int32)
    for i in range(n):
        if not np.isfinite(pos[i]).all():
            continue
        d2 = dist2(np.broadcast_to(pos[i], pos.shape), pos)
        js = np.flatnonzero((d2 < r * r) & (np.arange(n) != i))
        js = js[np.lexsort((js, d2[js]))]
        count[i] = len(js)
        for m, j in enumerate(js[:k]):
            idx[i, m] = j
            rows[i, 6 * m:6 * m + 3] = pos[j] - pos[i]
            rows[i, 6 * m + 3:6 * m + 6] = vel[j] - vel[i]
    return idx, rows, count


def assert_same(got, want, what=""):
    for name, g, w in zip(("idx", "rows", "count"), got, want):
        assert g.shape == w.shape, f"{what} {name}: shape {g.shape} != {w.shape}"
        if not np.array_equal(g, w):
            bad = np.argwhere(g != w) if g.ndim == 1 else np.argwhere((g != w).any(axis=1))
            raise AssertionError(f"{what} {name}: {len(bad)} rows differ, first {bad[:5].ravel().tolist()}")


def clustered(n, r, seed, offset=0.0):
    """Clusters of about 250 UAVs with a spread of r: tens of neighbours per UAV in the cores, few at the fringes."""
    rng = np.random.default_rng(seed)
    n_cl = max(1, n // 250)
    side = 10.0 * r * n_cl ** (1 / 3)
    centres = rng.uniform(0, side, (n_cl, 3))
    pos = centres[rng.integers(0, n_cl, n)] + rng.normal(0, r, (n, 3)) + offset
    vel = rng.normal(0, 2.0, (n, 3))
    return pos, vel


def test_reference_equals_brute_force():
    """n = 300: a unit lattice (equal distances everywhere), coincident UAVs, a dense clump (counts above k), non-finite rows."""
    rng = np.random.default_rng(5)
    g = np.stack(np.meshgrid(np.arange(5.0), np.arange(5.0), np.arange(4.0), indexing="ij"), -1).reshape(-1, 3)  # 100
    clump = rng.normal(0, 0.8, (120, 3)) + 20.0
    spread = rng.uniform(-5, 30, (74, 3))
    pos = np.concatenate([g, clump, spread, g[:3], clump[:3]])  # 300, six of them coincident with another
    pos[290] = [np.nan, 0, 0]
    pos[291] = [0, np.inf, 0]
    vel = rng.normal(0, 1, pos.shape)
    assert len(pos) == 300
    for r, k in ((1.0, 4), (1.5, 8), (2.0, 16), (2.5, 3)):
        want = brute_force(pos, vel, r, k)
        assert_same(reference(pos, vel, r, k), want, f"r={r} k={k}")
        assert want[2].max() > k and (want[0] >= 0).sum() > 0
    _, _, cnt = brute_force(pos, vel, 1.0, 4)
    assert cnt[290] == cnt[291] == 0


# ---- GPU ----------------------------------------------------------------------------------------------


def Batch(*a, **kw):
    from mrs_multirotor_simulator_b200 import UavBatch

    return UavBatch(*a, **kw)


def af(name, **kw):
    from mrs_multirotor_simulator_b200 import airframe

    return airframe(name, **kw)


def gpu_neighbours(b, r, k, stride=None, outputs=("idx", "rows", "count"), fill=7):
    import torch

    n, w = b.n, 6 * k if stride is None else stride
    dev = torch.device("cuda:0")
    idx = torch.full((n, k), -fill, dtype=torch.int32, device=dev)
    rows = torch.full((n, w), float(fill), dtype=torch.float64, device=dev)
    cnt = torch.full((n,), -fill, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    b.pack_neighbours_device(r, k, idx.data_ptr() if "idx" in outputs else None, rows.data_ptr() if "rows" in outputs else None,
                             cnt.data_ptr() if "count" in outputs else None, stride)
    b.sync()
    return idx.cpu().numpy(), rows.cpu().numpy(), cnt.cpu().numpy()


def check_against_state(b, radii_k, what=""):
    """The call on b against the reference on b's state (positions and velocities from get_state)."""
    st = b.get_state(fields=("x", "v"))
    for r, k in radii_k:
        want = reference(st["x"], st["v"], r, k)
        assert_same(gpu_neighbours(b, r, k), want, f"{what} r={r} k={k}")
    return want


def batch_at(pos, vel, types=None, tou=None):
    n = len(pos)
    b = Batch(types or [af("x500")], type_of_uav=tou, spawn_xyz=np.nan_to_num(pos), n=n)
    b.set_state(x=pos, v=vel)
    return b


@pytest.mark.gpu
@pytest.mark.parametrize("n, r", [(400, 0.5), (400, 3.0), (400, 12.0), (65536, 0.5), (65536, 3.0), (65536, 12.0), (1048576, 3.0)])
def test_random_clustered_swarms(n, r):
    pos, vel = clustered(n, r, seed=int(10 * r) + n % 97)
    b = batch_at(pos, vel)
    idx, rows, cnt = reference(pos, vel, r, MAX_K)
    assert np.mean(cnt > MAX_K) > 0.3 and cnt.max() > 4 * MAX_K
    for k in (1, 8, 16):
        assert_same(gpu_neighbours(b, r, k), (idx[:, :k], rows[:, :6 * k], cnt), f"n={n} r={r} k={k}")


@pytest.mark.gpu
def test_bench_grid_after_six_seconds_of_flight():
    """The bench swarm (a 65,536-UAV slice of its grid, VelocityHdgRate commands, collisions on) flown 600 ticks: states from the
    stepping kernel, velocities of metres per second."""
    from bench import workload, x500_world
    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_RATE_CMD

    n = 65536
    spawn, cmd = workload(0, n)
    b = Batch([x500_world()], spawn_xyz=spawn, n=n)
    b.set_input(VELOCITY_HDG_RATE_CMD, cmd)
    b.set_collisions(True, False, 100.0)
    b.run(0.01, 600, with_collisions=True)
    _, _, cnt = check_against_state(b, [(2.0, 4), (5.0, 8), (10.0, 16)], "bench grid")
    assert cnt.mean() > 8


@pytest.mark.gpu
def test_bucketed_batch_in_the_callers_order():
    """x500 / f550 / naki interleaved by index: the tiled arrays hold them sorted by airframe; outputs are in external order."""
    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD

    n = 3 * 7001
    tou = (np.arange(n) % 3).astype(np.int32)
    pos, vel = clustered(n, 3.0, seed=11)
    pos[:, 2] += 40.0
    b = batch_at(pos, vel, [af("x500"), af("f550"), af("naki")], tou)
    assert b.device_view().slot_of_uav is not None
    b.set_input(VELOCITY_HDG_CMD, np.tile([0.5, -0.3, 0.2, 0.1], (n, 1)))
    b.make_step(0.01, 5)
    check_against_state(b, [(3.0, 16), (1.0, 5)], "bucketed")


def _lattice_and_edges(r):
    """A unit lattice with coincident copies (exact ties), and far apart pairs at distance r * (1 + t * 2^-52), t = -4..4, along the
    axes and diagonals, whose first UAV sits on or next to a cell boundary of either layout."""
    g = np.stack(np.meshgrid(np.arange(8.0), np.arange(8.0), np.arange(3.0), indexing="ij"), -1).reshape(-1, 3)
    pts = [g, g[::7]]  # 192 + 28: the edge pairs start at index 220
    dirs = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 0], [1, 0, 1], [1, 1, 1], [-1, 0, 0], [0, -1, -1]], dtype=np.float64)
    dirs /= np.linalg.norm(dirs, axis=1)[:, None]
    reach = r * (1 + 2.0 ** -20)
    slot = 0
    for cell in (reach, 2 * reach, r, 2 * r):
        for m in (-3, -1, 1, 2, 5):
            for e in (-2, -1, 0, 1, 2):
                base = m * cell + e * np.spacing(m * cell)
                for d in dirs:
                    for t in range(-4, 5):
                        q = np.array([base, 50.0 * r * (slot % 40) + base, 30.0 * r * (slot // 40) + 100.0])
                        pts.append(np.stack([q, q + d * (r * (1 + t * 2.0 ** -52))]))
                        slot += 1
    return np.concatenate(pts)


@pytest.mark.gpu
@pytest.mark.parametrize("r", [0.5, 2.0, 3.0])
def test_ties_coincident_uavs_and_the_radius_edge(r):
    pos = _lattice_and_edges(r)
    vel = np.random.default_rng(3).normal(0, 1, pos.shape)
    b = batch_at(pos, vel)
    st = b.get_state(fields=("x", "v"))
    assert np.array_equal(st["x"], pos)
    idx, rows, cnt = reference(pos, vel, r, MAX_K)
    assert_same(gpu_neighbours(b, r, MAX_K), (idx, rows, cnt), f"r={r}")
    # both sides of the edge are exercised: pairs just inside and just outside the radius
    d2 = dist2(pos[220::2], pos[221::2])
    assert (d2 < r * r).sum() > 100 and (d2 >= r * r).sum() > 100


@pytest.mark.gpu
@pytest.mark.parametrize("r, offset", [(0.5, -4.0e8), (0.5, 3.0e8), (3.0, -2.5e9), (3.0, 3.0e9), (12.0, 1.0e10)])
def test_large_coordinates_inside_the_documented_range(r, offset):
    assert abs(offset) + 100 * r < 2.0 ** 30 * r
    pos, vel = clustered(20000, r, seed=7, offset=offset)
    pos[::3, 0] = -pos[::3, 0]  # both signs on one axis
    b = batch_at(pos, vel)
    want = reference(pos, vel, r, 8)
    assert want[2].mean() > 8
    assert_same(gpu_neighbours(b, r, 8), want, f"offset {offset}")


@pytest.mark.gpu
def test_stencil_row_across_the_end_of_the_bucket_table():
    """x-adjacent cells whose buckets are B-1 and 0, found through the mirror buckets.  The cell edge (2 * reach) and the table
    size (1024 buckets below 683 UAVs) follow api.cu / collide.cu; were they to change, the comparison still holds."""
    from test_collisions_gpu import _row_hash

    r = 1.0
    cell, n_buckets = 2 * r * (1 + 2.0 ** -20), 1024
    hits = []
    for cy in range(-40, 40):
        for cz in range(0, 4):
            cx = (n_buckets - 1 - _row_hash(cy, cz)) % n_buckets
            if cx < 200:
                hits.append((cx, cy, cz))
    assert len(hits) >= 8
    pts = []
    for cx, cy, cz in hits[:40]:
        xb = cell * (cx + 1)
        y, z = cell * cy + 0.5 * cell, cell * cz + 0.5 * cell
        pts += [[xb - 0.3, y, z], [xb + 0.3, y, z], [xb + 0.6, y + 0.1, z], [xb - 0.9, y - 0.2, z], [xb + 1.5, y, z]]
    pos = np.array(pts)
    vel = np.random.default_rng(4).normal(0, 1, pos.shape)
    b = batch_at(pos, vel)
    want = reference(pos, vel, r, 4)
    assert want[2].sum() >= 4 * len(hits[:40])
    assert_same(gpu_neighbours(b, r, 4), want, "wrap")


@pytest.mark.gpu
def test_non_finite_positions_have_no_neighbours_and_are_nobodys():
    pos, vel = clustered(4000, 2.0, seed=9)
    b = batch_at(pos, vel)
    bad = np.array([3, 17, 18, 400], dtype=np.int32)
    x = pos[bad].copy()
    x[0, 0], x[1, 1], x[2, 2], x[3] = np.nan, np.inf, -np.inf, [np.inf, np.nan, 1.0]
    b.set_state(idx=bad, x=x)
    st = b.get_state(fields=("x", "v"))
    assert not np.isfinite(st["x"][bad]).all(axis=1).any()
    want = reference(st["x"], st["v"], 2.0, 16)
    got = gpu_neighbours(b, 2.0, 16)
    assert_same(got, want, "non-finite")
    assert (got[2][bad] == 0).all() and not np.isin(got[0], bad).any()


@pytest.mark.gpu
def test_reads_the_state_not_the_packed_positions():
    """Collisions off and no optional outputs; then positions written by respawn_masked_device, set_state and through the device
    view, each without publish_positions: the call sees the new positions every time."""
    import torch
    from cuda.bindings import runtime as cudart
    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD

    n, r = 8192, 3.0
    pos, vel = clustered(n, r, seed=21)
    pos[:, 2] += 30.0
    plain = batch_at(pos, vel)
    quiet = batch_at(pos, vel)
    quiet.set_outputs(imu=False, positions=False)
    quiet.set_collisions(False, False, 0.0)
    for b in (plain, quiet):
        b.set_input(VELOCITY_HDG_CMD, np.tile([1.0, 0.5, 0.0, 0.0], (n, 1)))
        b.make_step(0.01, 20)
    assert np.array_equal(plain.get_state()["x"], quiet.get_state()["x"])
    want = check_against_state(quiet, [(r, 8)], "outputs off")
    assert_same(gpu_neighbours(plain, r, 8), want, "plain")

    b = quiet
    dev = torch.device("cuda:0")
    mask = torch.zeros(n, dtype=torch.bool, device=dev)
    mask[::5] = True
    xyz = torch.as_tensor(pos[::-1].copy() + [7.0, 0.0, 0.0], device=dev)
    hdg = torch.zeros(n, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    b.respawn_masked_device(mask.data_ptr(), xyz.data_ptr(), hdg.data_ptr())
    check_against_state(b, [(r, 8)], "after respawn_masked_device")

    sel = np.arange(1, n, 7, dtype=np.int32)
    b.set_state(idx=sel, x=pos[sel] + [0.0, -2.0, 1.0], v=np.ones((len(sel), 3)))
    check_against_state(b, [(r, 8)], "after set_state")

    v = b.device_view()
    st = np.empty((n // 128, 18, 128))
    (err,) = cudart.cudaMemcpy(st.ctypes.data, v.state, st.nbytes, cudart.cudaMemcpyKind.cudaMemcpyDeviceToHost)
    assert err == cudart.cudaError_t.cudaSuccess
    st[:, 0, :] += 1.5  # x of every UAV, rows 0-2 of the tiled state
    st[3, 1, :] = st[0, 1, :]  # tile 3 onto tile 0 in y
    (err,) = cudart.cudaMemcpy(v.state, st.ctypes.data, st.nbytes, cudart.cudaMemcpyKind.cudaMemcpyHostToDevice)
    assert err == cudart.cudaError_t.cudaSuccess
    check_against_state(b, [(r, 8)], "after a write through the device view")


@pytest.mark.gpu
def test_the_collision_pass_does_not_see_the_call():
    """Twin handles, collisions and neighbour lists on, 300 single-tick runs; one of them packs neighbours every tick."""
    from bench import workload, x500_world
    from mrs_multirotor_simulator_b200 import VELOCITY_HDG_RATE_CMD
    import torch

    n = 16384
    spawn, cmd = workload(0, n)
    spawn[:, 1] -= 1.8 * ((np.arange(n) // 1024) % 2)  # rows 2.2 m apart: pairs collide from the start
    twins = []
    for _ in range(2):
        b = Batch([x500_world()], spawn_xyz=spawn, n=n)
        b.set_input(VELOCITY_HDG_RATE_CMD, cmd)
        b.set_collisions(True, False, 100.0)
        twins.append(b)
    a, c = twins
    assert a.collision_info()["neighbour_lists"]
    idx = torch.empty((n, 8), dtype=torch.int32, device="cuda:0")
    rows = torch.empty((n, 48), dtype=torch.float64, device="cuda:0")
    cnt = torch.empty(n, dtype=torch.int32, device="cuda:0")
    pairs_seen = 0
    for tick in range(300):
        a.pack_neighbours_device(4.0, 8, idx.data_ptr(), rows.data_ptr(), cnt.data_ptr())
        for b in twins:
            b.run(0.01, 1, with_collisions=True)
        if tick % 30 == 29:
            pa, pc = a.get_collision_pairs(), c.get_collision_pairs()
            assert np.array_equal(pa, pc), f"tick {tick}"
            pairs_seen += len(pa)
    assert pairs_seen > 0
    sa, sc = a.get_full_state(), c.get_full_state()
    for key in sa:
        assert np.array_equal(sa[key], sc[key]), key
    assert np.array_equal(a.get_force(), c.get_force())
    assert np.array_equal(a.has_crashed(), c.has_crashed())
    ia, ic = a.collision_info(), c.collision_info()
    assert (ia["passes"], ia["rebuilds"]) == (ic["passes"], ic["rebuilds"]) and ia["rebuilds"] > 1
    ca, cc = a.counters(), c.counters()
    assert [ca[k] for k in ("steps", "collision_passes", "pairs", "crashed")] == [cc[k] for k in ("steps", "collision_passes", "pairs", "crashed")]
    assert ca["launches"] == cc["launches"] + 300 * 5
    st = a.get_state(fields=("x", "v"))
    a.pack_neighbours_device(4.0, 8, idx.data_ptr(), rows.data_ptr(), cnt.data_ptr())
    a.sync()
    assert_same((idx.cpu().numpy(), rows.cpu().numpy(), cnt.cpu().numpy()), reference(st["x"], st["v"], 4.0, 8), "twin")


@pytest.mark.gpu
def test_null_outputs_and_a_wider_stride():
    pos, vel = clustered(5000, 2.0, seed=13)
    b = batch_at(pos, vel)
    k = 6
    idx, rows, cnt = reference(pos, vel, 2.0, k)
    for outs in (("idx",), ("rows",), ("count",), ("idx", "count"), ("rows", "count")):
        gi, gr, gc = gpu_neighbours(b, 2.0, k, outputs=outs, fill=7)
        assert np.array_equal(gi, idx) if "idx" in outs else (gi == -7).all()
        assert np.array_equal(gr, rows) if "rows" in outs else (gr == 7.0).all()
        assert np.array_equal(gc, cnt) if "count" in outs else (gc == -7).all()
    gi, gr, gc = gpu_neighbours(b, 2.0, k, stride=6 * k + 5, fill=7)
    assert_same((gi, gr[:, :6 * k], gc), (idx, rows, cnt), "stride 6k+5")
    assert (gr[:, 6 * k:] == 7.0).all()


@pytest.mark.gpu
def test_invalid_arguments():
    import torch

    from mrs_multirotor_simulator_b200 import _lib

    L = _lib.lib()
    b = batch_at(*clustered(300, 1.0, seed=1))
    buf = torch.zeros((300, 6 * 17), dtype=torch.float64, device="cuda:0")
    ib = torch.zeros((300, 17), dtype=torch.int32, device="cuda:0")
    cb = torch.zeros(300, dtype=torch.int32, device="cuda:0")
    p, q = buf.data_ptr(), ib.data_ptr()

    def rc(radius, k, idx, rows, stride, count):
        return L.mrsb_pack_neighbours_device(b.h, radius, k, idx, rows, stride, count)

    for radius in (float("nan"), float("inf"), -float("inf"), 0.0, -1.0, -0.0):
        assert rc(radius, 4, q, p, 24, None) == ERR_INVALID, radius
    for k in (0, -1, 17, 1 << 20):
        assert rc(1.0, k, q, p, 6 * 17, None) == ERR_INVALID, k
    assert rc(1.0, 4, None, p, 23, None) == ERR_INVALID
    assert rc(1.0, 4, q, None, 0, None) == 0  # the stride only matters with rows
    assert rc(1.0, 4, None, None, 24, None) == ERR_INVALID
    assert rc(1.0, 16, q, p, 96, cb.data_ptr()) == 0
    assert L.mrsb_pack_neighbours_device(None, 1.0, 4, q, p, 24, None) == ERR_INVALID
    sharded = Batch([af("x500")], spawn_xyz=np.zeros((4, 3)), n=4, n_global=8, shard_begin=4)
    assert L.mrsb_pack_neighbours_device(sharded.h, 1.0, 4, q, p, 24, None) == ERR_STATE
    assert L.mrsb_pack_neighbours_device(sharded.h, 0.0, 4, q, p, 24, None) == ERR_INVALID
    b.sync()


@pytest.mark.gpu
def test_repeated_calls_allocate_nothing():
    import torch

    n = 1 << 18
    b = batch_at(*clustered(n, 2.0, seed=17))
    rows = torch.empty((n, 96), dtype=torch.float64, device="cuda:0")
    b.pack_neighbours_device(2.0, 16, rows_ptr=rows.data_ptr())
    b.sync()
    free0 = torch.cuda.mem_get_info(0)[0]
    for k in range(20):
        b.pack_neighbours_device(0.5 + k, 1 + k % 16, rows_ptr=rows.data_ptr())
    b.sync()
    # a workspace allocated again would take about 136 bytes per UAV (36 MB); the device is shared, so allow for others' noise
    assert free0 - torch.cuda.mem_get_info(0)[0] < 16 << 20


@pytest.mark.gpu
def test_returns_while_a_long_stepping_launch_runs():
    import torch
    from cuda.bindings import runtime as cudart

    n = 1 << 20
    b = batch_at(*clustered(n, 2.0, seed=19))
    cnt = torch.empty(n, dtype=torch.int32, device="cuda:0")
    b.pack_neighbours_device(2.0, 8, count_ptr=cnt.data_ptr())  # the workspace exists from here on
    b.sync()
    b.make_step(0.01, 1000)
    b.pack_neighbours_device(2.0, 8, count_ptr=cnt.data_ptr())
    (err,) = cudart.cudaStreamQuery(b.stream)
    assert err == cudart.cudaError_t.cudaErrorNotReady
    b.sync()
