#!/usr/bin/env python
"""bench.py — UAV-steps/s of the stepping path (RK4 + controller cascade + collisions).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port +
                                                             # the real vendored nanoflann), all host threads
    python bench.py --gpus 1 ... --dump-outputs DIR          # also writes what the timed path computed in its
                                                             # last tick as DIR/<name>.npy (see dump_outputs)

Workload (BASELINE.json config 4 = the configuration the metric is quoted on):
  1,048,576 x500 UAVs on a 1024 x 1024 grid, 4 m pitch, spawned at z = 0, heading 0; world of
  config/multirotor_simulator.yaml (dt = 0.01 s, g = 9.81, ground plane at z = 0, collisions on,
  crash:false, rebounce 100 as in tmux/standalone_400_uavs); two 0.01 s zero-actuator warm-up steps
  (uav_system_ros.cpp:223-232); seeded VelocityHdgRate commands v_xy~U(-2,2), v_z~U(0,2),
  hdg_rate~U(-1,1) (tmux/standalone_400_uavs/velocity_cmd.py:33-39) from the counter RNG of SURVEY
  §8d; K = 1 (collisions every step).  One "step" = one tick of the reference node's loop
  (multirotor_simulator.cpp:198-231): makeStep for every UAV, then handleCollisions.
  With N GPUs the SAME 1 Mi swarm is sharded by contiguous index ranges (strong scaling); the collision
  pass of a shard pulls the positions it needs from its peers' memory over NVLink.

What is timed.  A swarm that has just been spawned on its grid has no UAV within reach of another: the
collision pass finds empty neighbour lists and never rebuilds its table — the cheapest ticks there are.
So the swarm is first flown untimed for --fast-forward ticks (default 600 = 6 s: UAVs have mixed, a third
of them has neighbours to check, pairs collide every tick, the spatial hash is rebuilt on ~6 % of the
ticks); then --reps (10) blocks of exactly --steps ticks are timed, each block bracketed by a barrier +
synchronize on both sides and driven by ONE mrsb_run call; `value` is the MEDIAN block (max over ranks
within a block); the fastest block and the fresh-grid figure are reported beside it
(`regimes`).  One JSON line on stdout (rank 0).  `value` is device-timed with inputs resident in HBM;
`e2e` goes through the public C ABI with pinned HOST buffers (commands in, positions out, every step).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the bench leaves the source tree as it found it (it may be read-only)

N_UAVS = 1 << 20
DT = 0.01
SEED = 42
METRIC = "UAV-steps/s (RK4+control+collisions) at 1M UAVs"
UNIT = "UAV-steps/s"
L2_BYTES = 126 * (1 << 20)
# algorithmic HBM bytes per UAV-step of the stepping kernel (SURVEY §8d): R = 144 + 8n + P + 24 + 8 + 4 + C, W = 144 + 8n + P
# (+24 when the IMU acceleration is exported).  VelocityHdg(Rate), quad: n = 4, P = 144, C = 32 -> 708 (+24);
# PositionCmd: P = 192 -> 804; ActuatorCmd: P = 0, C = 8n -> 420 / 468 / 516 for n = 4 / 6 / 8.
STEP_BYTES_VELOCITY_QUAD = 708
IMU_BYTES = 24
ACTUATOR_BYTES = {4: 420, 6: 468, 8: 516}
# as-written FP64 census of the reference for these modes (SURVEY §8d)
STEP_FLOP_VELOCITY_QUAD = 2550
COLLIDE_BYTES_PER_UAV = 52


def u01(seed, stream, index):
    with np.errstate(over="ignore"):
        g = np.uint64(0x9E3779B97F4A7C15)
        z = np.uint64(seed) + g * ((np.uint64(stream) << np.uint64(32)) + np.asarray(index, dtype=np.uint64))
        z = z + g
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def workload(begin, count, side=1024):
    """Spawn positions and commands of UAVs [begin, begin+count) of the 1 Mi swarm."""
    k = np.arange(begin, begin + count)
    spawn = np.stack([4.0 * (k % side), 4.0 * (k // side), np.zeros(count)], axis=1).astype(np.float64)
    cmd = np.stack([-2 + 4 * u01(SEED, 1, k), -2 + 4 * u01(SEED, 2, k), 2 * u01(SEED, 3, k), -1 + 2 * u01(SEED, 4, k)], axis=1)
    return spawn, np.ascontiguousarray(cmd)


DUMP_ROWS = 65536       # UAVs whose whole state --dump-outputs writes (positions: every UAV)
DUMP_MAX_PAIRS = 1 << 21


def seeded_sample(count, k, stream):
    """`k` of range(count), sorted: the ones with the smallest counter-RNG draws (the same on every run and numpy version)."""
    return np.sort(np.argsort(u01(SEED, stream, np.arange(count)), kind="stable")[:k])


def dump_outputs(out_dir, batch, x):
    """Writes what a caller of the timed path (mrsb_run: makeStep for every UAV, then handleCollisions) receives after its last
    tick, one .npy per array: x = every UAV's position; <field>_sample = the whole state, IMU acceleration and collision force
    of DUMP_ROWS seeded UAVs (their indices in sample_rows); collision_pairs = the directed (i, j) pairs of the last pass, in
    float32 (indices < 2^24 are exact), a seeded sample of DUMP_MAX_PAIRS when there are more.  At most 60 MB in all."""
    os.makedirs(out_dir, exist_ok=True)
    rows = seeded_sample(len(x), DUMP_ROWS, 100).astype(np.int32)
    out = {"x": x, "sample_rows": rows.astype(np.float64)}
    for k, a in batch.get_full_state(rows).items():
        if k != "x":
            out[f"{k}_sample"] = a
    out["force_sample"] = batch.get_force(rows)
    pairs = batch.get_collision_pairs()
    if len(pairs) > DUMP_MAX_PAIRS:
        pairs = pairs[seeded_sample(len(pairs), DUMP_MAX_PAIRS, 101)]
    out["collision_pairs"] = pairs.astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def x500_world():
    from mrs_multirotor_simulator_b200 import airframe

    return airframe("x500", ground_enabled=True, ground_z=0.0, takeoff_patch_enabled=False, g=9.81)


def checksum(a):
    """64-bit checksum of the raw bytes of a float64 array: the wrapping sum of its uint64 words (additive over shards)."""
    return int(np.ascontiguousarray(a, dtype=np.float64).view(np.uint64).sum(dtype=np.uint64))


def combine_checksums(cs, dist, device=None):
    """The swarm's checksum from the shards': the wrapping sum over ranks (a uint64 travels as two int64 words)."""
    import torch

    t = torch.tensor([cs & 0x7FFFFFFFFFFFFFFF, cs >> 63], dtype=torch.int64, device=device)
    parts = [torch.zeros_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t)
    return sum(int(p[0].item()) | (int(p[1].item()) << 63) for p in parts) & 0xFFFFFFFFFFFFFFFF


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        self.f.seek(0)
        sm, mx, power, reasons = [], [], [], set()
        for line in self.f.read().splitlines():
            c = [t.strip() for t in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
                power.append(float(c[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = [s for s, p in zip(sm, power) if p >= 0.5 * max(power)] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": float(max(power))}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def workload_config(n_gpus):
    """Identical in both arms (the driver compares them)."""
    # bytes one tick touches per GPU: the stepping kernel's algorithmic traffic (each byte read once or written once) + the collision pass'
    working_set = (N_UAVS // n_gpus) * (STEP_BYTES_VELOCITY_QUAD + IMU_BYTES + COLLIDE_BYTES_PER_UAV)
    l2 = ("L2 flushed between timed steps (256 MiB memset, outside the event pairs)" if working_set < L2_BYTES else
          f"per-GPU working set {working_set / 1e6:.0f} MB per tick > 126 MB L2: inputs larger than L2, no flush")
    return {"workload": "C4: 1,048,576 x500 UAVs, 1024x1024 grid 4 m pitch, VelocityHdgRate commands, dt=0.01, K=1, ground plane + mutual collisions "
                        "(rebounce 100) every tick", "n_uavs": N_UAVS, "dt": DT, "k_substeps": 1, "collisions": "enabled, crash=false, rebounce=100",
            "sharding": f"{n_gpus} contiguous index shards (strong scaling), cross-shard neighbours read from the owning GPU every tick" if n_gpus > 1 else "single shard",
            "l2": l2}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU path on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference(n_sample, ticks, warmup, threads, fast=False, fast_forward=0):
    """Times `ticks` ticks (makeStep for all + handleCollisions) of the CPU path on the first `n_sample` UAVs of the workload:
    oracle port for UavSystem::makeStep (the reference itself needs Eigen + Boost, absent from the image), the REAL vendored
    nanoflann for handleCollisions.  Returns (UAV-steps/s, ms per tick, description)."""
    from oracle import binding as O

    spawn, cmd = workload(0, n_sample)
    cls = O.FastOracleSwarm if fast else O.OracleSwarm
    sw = cls([x500_world()], spawn_xyz=spawn, n=n_sample)
    sw.set_input(O.ACTUATOR_CMD, np.zeros((n_sample, 8)))
    sw.make_step(DT, 2, threads)
    sw.set_input(O.VELOCITY_HDG_RATE_CMD, cmd)
    sw.set_collisions(True, False, 100.0)
    engine = "nanoflann" if O.ref_lib() is not None else "port"
    for _ in range(warmup + fast_forward):
        sw.make_step(DT, 1, threads)
        sw.handle_collisions(engine=engine, n_threads=threads, cap=1 << 16)
    t0 = time.perf_counter()
    for _ in range(ticks):
        sw.make_step(DT, 1, threads)
        sw.handle_collisions(engine=engine, n_threads=threads, cap=1 << 16)
    dt = time.perf_counter() - t0
    what = "the whole 1 Mi swarm" if n_sample == N_UAVS else f"{n_sample} UAVs (first rows of the 1 Mi grid)"
    desc = (f"{what} x {ticks} ticks after {warmup + fast_forward} untimed ones, {threads} threads; stepping = oracle port "
            f"({'-O3 -march=native, built on this host' if fast else '-O2 -ffp-contract=off: the parity build'}), collisions = "
            f"{'real vendored nanoflann (KD-tree build 1 thread, queries threaded)' if engine == 'nanoflann' else 'cell-list port'}")
    return n_sample * ticks / dt, dt / ticks * 1e3, desc


_PORT_CHECK = None


def port_vs_reference_sources(n=2048, ticks=20):
    """The timed port against the reference's OWN UavSystem sources compiled against the Eigen/odeint stand-ins
    (oracle/_ref/libref_uavsystem.so, built where /root/reference exists and shipped): same bits, and how fast each is."""
    global _PORT_CHECK
    if _PORT_CHECK is None:
        from oracle import binding as O

        if O.refsys_lib() is None:
            _PORT_CHECK = "reference-sources build (oracle/_ref/libref_uavsystem.so) not shipped: port not re-verified in this run"
        else:
            spawn, cmd = workload(0, n)
            rate = {}
            state = {}
            for name, cls in (("port", O.OracleSwarm), ("reference sources", O.RefSwarm)):
                sw = cls([x500_world()], spawn_xyz=spawn, n=n)
                sw.set_input(O.VELOCITY_HDG_RATE_CMD, cmd)
                t0 = time.perf_counter()
                sw.make_step(DT, ticks, 1)
                rate[name] = n * ticks / (time.perf_counter() - t0)
                state[name] = sw.get_state()
            same = all(np.array_equal(state["port"][k], state["reference sources"][k]) for k in state["port"])
            _PORT_CHECK = (f"port {'bit-identical to' if same else 'DIFFERS from'} the reference's own UavSystem sources compiled against Eigen/odeint stand-ins "
                           f"on {n} UAVs x {ticks} ticks (1 thread: port {rate['port'] / 1e6:.2f} M, reference sources {rate['reference sources'] / 1e6:.2f} M UAV-steps/s; "
                           f"the faster one is the baseline)")
    return _PORT_CHECK


def run_reference(args):
    """The reference arm on the metric's own configuration: the WHOLE 1 Mi swarm, every tick = makeStep for all + the real
    nanoflann pass, all host threads.  A tick takes ~0.3 s on 16 threads, so --steps 20 --warmup 5 runs ~10 s; larger step
    counts are cut to what fits ~3 minutes (said in `sample`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    speed, _, _ = cpu_reference(65536, 2, 1, threads)
    budget_ticks = max(3, int(150.0 * speed / N_UAVS))
    warmup = min(args.warmup, max(1, budget_ticks // 5))
    ticks = max(1, min(args.steps, budget_ticks - warmup))
    value, ms, desc = cpu_reference(N_UAVS, ticks, warmup, threads)
    if ticks != args.steps:
        desc += f"; --steps {args.steps} cut to {ticks} timed ticks to stay within minutes"
    desc += "; " + port_vs_reference_sources()
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


EXCHANGE = {0: "none (single shard)", 1: "NCCL all-gather of packed xyz per tick",
            2: "pull over peer memory (CUDA IPC + NVLink): hand-shake per tick, each shard fetches its halo's positions from the owners"}


# ------------------------------------------------------------------------------------------------
# parity record carried by the bench line
# ------------------------------------------------------------------------------------------------
def parity_record(device, ticks=300, n=65536):
    """The first 64 rows of the bench swarm (65,536 UAVs: enough tiles for the persistent staged kernel that `value` times) flown from
    spawn on the GPU and in the CPU oracle (real nanoflann collision loop) with the bench's commands: state differences after `ticks`
    ticks, and the directed collision pair lists compared on every tick."""
    from mrs_multirotor_simulator_b200 import ACTUATOR_CMD, VELOCITY_HDG_RATE_CMD, UavBatch
    from oracle import binding as O

    threads = os.cpu_count() or 1
    spawn, cmd = workload(0, n)
    # denser than the bench grid along y so that collisions happen within the first seconds: every second row shifted towards its neighbour
    spawn[:, 1] -= 1.8 * ((np.arange(n) // 1024) % 2)
    gpu = UavBatch([x500_world()], spawn_xyz=spawn, n=n, device=device)
    orc = O.OracleSwarm([x500_world()], spawn_xyz=spawn, n=n)
    engine = "nanoflann" if O.ref_lib() is not None else "port"
    for s in (gpu, orc):
        s.set_input(ACTUATOR_CMD, np.zeros((n, 8)))
    gpu.make_step(DT)
    gpu.make_step(DT)
    orc.make_step(DT, 2, threads)
    for s in (gpu, orc):
        s.set_collisions(True, False, 100.0)
        s.set_input(VELOCITY_HDG_RATE_CMD, cmd)
    gpu.set_pair_capacity(1 << 18)
    pairs_total, pairs_equal, first_diff = 0, True, None
    for t in range(ticks):
        gpu.make_step(DT)
        gpu.handle_collisions()
        orc.make_step(DT, 1, threads)
        po = orc.handle_collisions(engine=engine, n_threads=threads, cap=1 << 18)
        pg = gpu.get_collision_pairs()
        po = po[np.lexsort((po[:, 1], po[:, 0]))] if len(po) else po.reshape(0, 2)
        pairs_total += len(po)
        if pairs_equal and not np.array_equal(po, pg):
            pairs_equal, first_diff = False, t
    variant = gpu.step_info()
    so, sg = orc.get_state(), gpu.get_full_state()
    out = {"n_uavs": n, "ticks": ticks, "kernel": f"{variant['variant']} <{variant['n_motors']} motors, mode {variant['mode']}>", "oracle_collisions": engine,
           "max_dx": float(np.max(np.abs(so["x"] - sg["x"]))), "max_dv": float(np.max(np.abs(so["v"] - sg["v"]))),
           "max_dR": float(np.max(np.abs(so["R"] - sg["R"]))), "max_domega": float(np.max(np.abs(so["omega"] - sg["omega"]))),
           "max_drpm": float(np.max(np.abs(so["motor_rpm"] - sg["motor_rpm"]))), "pairs_total": int(pairs_total), "pairs_equal": bool(pairs_equal),
           "tolerance": {"x": 1e-9, "v": 1e-9, "R": 1e-10, "omega": 1e-8, "motor_rpm": 1e-6}}
    if first_diff is not None:
        out["first_tick_with_different_pairs"] = first_diff
    out["within_tolerance"] = bool(out["max_dx"] <= 1e-9 and out["max_dv"] <= 1e-9 and out["max_dR"] <= 1e-10 and out["max_domega"] <= 1e-8 and
                                   out["max_drpm"] <= 1e-6)
    gpu.close()
    return out


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch

    from mrs_multirotor_simulator_b200 import ACTUATOR_CMD, VELOCITY_HDG_CMD, VELOCITY_HDG_RATE_CMD, UavBatch, _lib, airframe
    from mrs_multirotor_simulator_b200.sharding import connect, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run --nproc-per-node N")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    begin, n_local = shard_range(N_UAVS, world, rank)
    warmup = max(args.warmup, 3)
    L = _lib.lib()
    cfg = workload_config(world)
    flush = cfg["l2"].startswith("L2 flushed")
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if flush else None

    def make_swarm():
        spawn, cmd = workload(begin, n_local)
        b = UavBatch([x500_world()], spawn_xyz=spawn, n=n_local, device=local, n_global=N_UAVS, shard_begin=begin)
        if world > 1:
            connect(b, dist)
        b.set_input(ACTUATOR_CMD, np.zeros((n_local, 8)))
        b.make_step(DT)
        b.make_step(DT)
        b.set_collisions(True, False, 100.0)
        b.set_input(VELOCITY_HDG_RATE_CMD, cmd)
        b.sync()
        return b, cmd

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_block(batch, stream, steps, run_fn=None, step_fn=None, flush=flush):
        """Exactly `steps` steps between a barrier + synchronize on both sides, timed with CUDA events on the handle's stream; returns
        ms (max over ranks).  Per-GPU working set above L2: ONE event pair around one call that issues all the steps (run_fn).
        Otherwise every step has its own pair and the L2 flush runs between the pairs."""
        barrier()
        if not flush:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            if run_fn is not None:
                run_fn(steps)
            else:
                for _ in range(steps):
                    step_fn()
            b.record(stream)
            barrier()
            ms = a.elapsed_time(b)
        else:
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for a, b in ev:
                with torch.cuda.stream(stream):
                    flush_buf.zero_()
                a.record(stream)
                if run_fn is not None:
                    run_fn(1)
                else:
                    step_fn()
                b.record(stream)
            barrier()
            ms = sum(a.elapsed_time(b) for a, b in ev)
        return max_over_ranks(ms)

    batch, cmd = make_swarm()
    stream = torch.cuda.ExternalStream(batch.stream, device=dev)
    run_ticks = lambda k: batch.run(DT, k, 1, True)

    # ---- regime "fresh_grid": the first ticks after spawn (nothing within reach of anything) ----
    run_ticks(warmup)
    info_a = batch.collision_info()
    fresh_steps = min(args.steps, 50)
    fresh_ms = timed_block(batch, stream, fresh_steps, run_fn=run_ticks) / fresh_steps
    info_b = batch.collision_info()
    fresh = {"ms_per_step": fresh_ms, "value": N_UAVS / (fresh_ms * 1e-3), "steps": fresh_steps,
             "rebuild_fraction": (info_b["rebuilds"] - info_a["rebuilds"]) / max(1, info_b["passes"] - info_a["passes"]), "pairs_last_tick": batch.counters()["pairs"]}

    # ---- fast-forward, untimed: the swarm mixes -------------------------------------------------
    done = warmup + fresh_steps
    if args.fast_forward > done:
        run_ticks(args.fast_forward - done)
    run_ticks(warmup)
    batch.sync()

    # ---- headline: --reps blocks of exactly --steps ticks in the mixed regime -------------------
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    c0 = batch.counters()["launches"]
    info0 = batch.collision_info()
    blocks = [timed_block(batch, stream, args.steps, run_fn=run_ticks) for _ in range(args.reps)]
    info1 = batch.collision_info()
    pairs_last = batch.counters()["pairs"]
    launches = (batch.counters()["launches"] - c0) / args.reps
    if sampler:
        clocks = sampler.stop()
    total_ms = float(np.median(blocks))
    value = N_UAVS * args.steps / (total_ms * 1e-3)
    ticks_flown = warmup + max(args.fast_forward, done) + warmup + args.reps * args.steps
    # the swarm every configuration of --gpus must have computed: checksum of all positions after the timed region
    x_now = batch.get_state(fields=("x",))["x"]
    cs = checksum(x_now)
    if dist is not None:
        cs = combine_checksums(cs, dist, dev)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, batch, x_now)

    # shards that fit into L2: the same blocks again without the flush between ticks (what a running simulation sees: tick t + 1
    # reads what tick t wrote), reported beside the headline
    resident = None
    if flush:
        rb = [timed_block(batch, stream, args.steps, run_fn=run_ticks, flush=False) for _ in range(args.reps)]
        resident = {"value": N_UAVS * args.steps / (float(np.median(rb)) * 1e-3), "ms_per_step": float(np.median(rb)) / args.steps, "blocks_ms": rb,
                    "note": "no L2 flush between ticks, one mrsb_run call per block"}

    # ---- roofline of the dominant kernel (the stepping kernel), timed alone ---------------------
    n_roof = min(max(args.steps, 50), 200)
    step_ms = timed_block(batch, stream, n_roof, step_fn=lambda: batch.make_step(DT, 1)) / n_roof
    step_info = batch.step_info()
    batch.set_outputs(imu=False, positions=True)
    step_ms_no_imu = timed_block(batch, stream, n_roof, step_fn=lambda: batch.make_step(DT, 1)) / n_roof
    batch.set_outputs(imu=True, positions=True)
    # a pass that is not preceded by exactly one stepping launch rebuilds the spatial hash: this times the rebuild pass
    coll_rebuild_ms = timed_block(batch, stream, min(n_roof, 50), step_fn=batch.handle_collisions) / min(n_roof, 50)
    # ... and a tick whose pass only checks the neighbour lists: the shortest of a run of single ticks
    singles = [timed_block(batch, stream, 1, run_fn=run_ticks) for _ in range(12)]
    list_tick_ms = float(np.min(singles))

    # ---- e2e: commands from pinned host memory in, positions to host out, every step -------------
    cmd_host = torch.from_numpy(cmd).pin_memory()
    pos_host = [torch.empty((n_local, 3), dtype=torch.float64).pin_memory() for _ in range(2)]

    def e2e_loop(n_ticks, pipelined, upload_every=1, out=None):
        """Every tick: VelocityHdgRate rows H2D (every `upload_every`-th tick), makeStep + handleCollisions (mrsb_run: one graph launch),
        positions D2H — through the C ABI.  pipelined: the upload of tick t+1 and the download of tick t-1 overlap tick t
        (mrsb_*_async); otherwise the blocking setInput/getState pair."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for t in range(n_ticks):
            if t % upload_every == 0:
                if pipelined:
                    _lib.check(L.mrsb_set_input_async(batch.h, VELOCITY_HDG_RATE_CMD, C.c_void_p(cmd_host.data_ptr()), 4))
                else:
                    _lib.check(L.mrsb_set_input_velocity_hdg_rate(batch.h, n_local, None, C.c_void_p(cmd_host.data_ptr())))
            _lib.check(L.mrsb_run(batch.h, DT, 1, 1, 1))
            if pipelined:
                _lib.check(L.mrsb_get_positions_async(batch.h, C.c_void_p((out or pos_host)[t & 1].data_ptr())))
            else:
                _lib.check(L.mrsb_get_state(batch.h, n_local, None, C.c_void_p(pos_host[0].data_ptr()), None, None, None, None))
        batch.sync()  # uploads, compute and downloads have all landed
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) * 1e-3)

    n_e2e = min(max(args.steps, 20), 200)
    e2e_loop(3, True)
    e2e_s = e2e_loop(n_e2e, True)
    last = pos_host[(n_e2e - 1) & 1].numpy().copy()
    # the downloaded positions are the simulation's: compare the last snapshot with a blocking read
    assert np.array_equal(last, batch.get_state(fields=("x",))["x"]), "e2e positions differ from a blocking read"
    e2e_10_s = e2e_loop(n_e2e, True, upload_every=10)
    # ... and a viewer that follows every fourth UAV only (mrsb_set_position_subset): commands on every 10th tick, 6.3 MB of positions per tick
    every4 = np.arange(0, n_local, 4, dtype=np.int32)
    batch.set_position_subset(every4)
    sub_host = [torch.empty((len(every4), 3), dtype=torch.float64).pin_memory() for _ in range(2)]
    e2e_loop(3, True, upload_every=10, out=sub_host)
    e2e_sub_s = e2e_loop(n_e2e, True, upload_every=10, out=sub_host)
    assert np.array_equal(sub_host[(n_e2e - 1) & 1].numpy(), batch.get_state(idx=every4, fields=("x",))["x"]), "subset download differs from a blocking read"
    batch.set_position_subset(None)
    e2e_loop(3, False)
    e2e_blocking_s = e2e_loop(min(n_e2e, 50), False)
    e2e_value = N_UAVS * n_e2e / e2e_s
    exchange = EXCHANGE[batch.exchange_mode()]
    batch.close()

    # ---- secondary configurations of BASELINE.json ----------------------------------------------
    secondary = []
    peaks, peak_kind = measured_peaks()
    fp64 = C.c_double()
    copy = C.c_double()
    L.mrsb_microbench_fp64(local, C.byref(fp64))
    L.mrsb_microbench_copy(local, C.byref(copy))
    ex_flop = None
    fp64_file = os.path.join(ROOT, "profiles", "step_kernel_fp64.json")
    if os.path.exists(fp64_file):  # executed FP64 work of the stepping kernel (ncu), reported beside the as-written census (SURVEY §8d)
        with open(fp64_file) as f:
            ex_flop = json.load(f)["executed_fp64_flop_per_uav_step"]

    if not args.no_secondary:
        # C5: 1 Mi UAVs, a third each x500 / f550 / naki interleaved by index, ActuatorCmd ~U(0.4, 0.7) re-drawn every 100 steps, ground
        # on, collisions off, sharded over the N GPUs (no exchange: nothing crosses shards without the collision pass)
        types = [airframe(f, ground_enabled=True, ground_z=0.0) for f in ("x500", "f550", "naki")]
        tou = (np.arange(N_UAVS) % 3).astype(np.int32)
        spawn, _ = workload(begin, n_local)
        b5 = UavBatch(types, type_of_uav=tou, spawn_xyz=spawn, n=n_local, device=local, n_global=N_UAVS, shard_begin=begin)
        b5.set_outputs(imu=True, positions=False)  # nothing consumes packed positions here: no collision pass, no position download
        st5 = torch.cuda.ExternalStream(b5.stream, device=dev)
        k = np.arange(begin, begin + n_local)
        # the two alternating command draws live on the device (an RL policy would produce them there): re-drawing = one
        # device-side scatter through mrsb_set_input_device, inside the timed region
        draws = [torch.from_numpy(np.ascontiguousarray(np.stack([0.4 + 0.3 * u01(SEED + d, 10 + m, k) for m in range(8)], axis=1))).to(dev) for d in range(2)]
        torch.cuda.synchronize()
        b5.set_input_device(ACTUATOR_CMD, draws[0].data_ptr(), 8)
        for _ in range(5):
            b5.make_step(DT)
        c5_steps = min(max(args.steps, 100), 200)
        c5_tick = [0]

        def c5_block(n):
            for _ in range(n):
                if c5_tick[0] % 100 == 0:
                    b5.set_input_device(ACTUATOR_CMD, draws[(c5_tick[0] // 100) & 1].data_ptr(), 8)
                b5.make_step(DT)
                c5_tick[0] += 1

        c5_ms = timed_block(b5, st5, c5_steps, run_fn=c5_block) / c5_steps
        info5 = b5.step_info()
        mean_bytes = sum(ACTUATOR_BYTES.values()) / 3 + IMU_BYTES
        secondary.append({"config": "C5: 1,048,576 UAVs, x500/f550/naki interleaved by index (4/6/8 motors), ActuatorCmd re-drawn every 100 steps (upload inside "
                                    "the timed region), ground on, collisions off, K=1", "n_gpus": world, "value": N_UAVS / (c5_ms * 1e-3), "unit": UNIT,
                          "ms_per_step": c5_ms, "steps": c5_steps, "kernel": f"{info5['variant']} <{info5['n_motors'] or 'per-UAV'} motors>",
                          "roofline": {"bound": "hbm", "achieved": n_local * mean_bytes / (c5_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                       "frac": n_local * mean_bytes / (c5_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes_per_uav_step": mean_bytes}})
        b5.close()
        if rank == 0:
            # C3: 65,536 x500 RL-style batch, random VelocityHdgCmd, K = 10 fused substeps per launch, 100 launches, 1 x B200
            n3 = 65536
            k3 = np.arange(n3)
            spawn3 = np.stack([4.0 * (k3 % 256), 4.0 * (k3 // 256), np.full(n3, 10.0)], axis=1)
            cmd3 = np.ascontiguousarray(np.stack([-2 + 4 * u01(SEED, 1, k3), -2 + 4 * u01(SEED, 2, k3), -2 + 4 * u01(SEED, 3, k3), -np.pi + 2 * np.pi * u01(SEED, 4, k3)], axis=1))
            b3 = UavBatch([airframe("x500")], spawn_xyz=spawn3, n=n3, device=local)
            st3 = torch.cuda.ExternalStream(b3.stream, device=dev)
            b3.set_input(VELOCITY_HDG_CMD, cmd3)
            for _ in range(5):
                b3.make_step(DT, 10)
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(100)]
            fb = flush_buf if flush_buf is not None else torch.empty(256 << 20, dtype=torch.uint8, device=dev)
            for a, e in ev:  # 65,536 UAVs fit in L2: flushed between launches
                with torch.cuda.stream(st3):
                    fb.zero_()
                a.record(st3)
                b3.make_step(DT, 10)
                e.record(st3)
            torch.cuda.synchronize()
            c3_ms = float(np.median([a.elapsed_time(e) for a, e in ev]))
            info3 = b3.step_info()
            tf_written = n3 * 10 * STEP_FLOP_VELOCITY_QUAD / (c3_ms * 1e-3) / 1e12
            r3 = {"bound": "fp64", "achieved": tf_written, "peak": fp64.value, "unit": "TFLOP/s (as-written census, 2550 flop per UAV-step)", "frac": tf_written / fp64.value,
                  "peak_source": "DFMA microbenchmark in this run (mrsb_microbench_fp64)"}
            if ex_flop:
                tf_ex = n3 * 10 * ex_flop / (c3_ms * 1e-3) / 1e12
                r3.update({"achieved_executed": tf_ex, "frac": min(tf_ex, tf_written) / fp64.value,
                           "note": "frac = the smaller of executed (ncu census) and as-written FP64 work over the measured DFMA peak (SURVEY §8d)"})
            secondary.append({"config": "C3: 65,536 x500, random VelocityHdgCmd, collisions and ground off, K=10 fused substeps per launch, 100 launches (L2 flushed between "
                                        "launches)", "n_gpus": 1, "value": n3 * 10 / (c3_ms * 1e-3), "unit": UNIT, "ms_per_launch": c3_ms,
                              "kernel": f"{info3['variant']} <{info3['n_motors']} motors, mode {info3['mode']}, K=10>", "roofline": r3})
            b3.close()

    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_record(local)

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    bytes_per_uav = STEP_BYTES_VELOCITY_QUAD + IMU_BYTES
    achieved = n_local * bytes_per_uav / (step_ms * 1e-3) / 1e9
    passes = max(1, info1["passes"] - info0["passes"])
    tick_ms = total_ms / args.steps
    roofline = {"kernel": f"uav_step_{step_info['variant']}_kernel<{step_info['n_motors']} motors, VELOCITY_HDG_RATE, K=1>", "bound": "hbm", "achieved": achieved,
                "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": None,
                "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                "algorithmic_bytes_per_uav_step": bytes_per_uav, "algorithmic_bytes_note": "SURVEY §8d: 708 B for VelocityHdg(Rate) quad + 24 B exported IMU acceleration",
                "launch_ms": step_ms, "uavs_per_launch": n_local,
                "imu_rows_off": {"launch_ms": step_ms_no_imu, "algorithmic_bytes_per_uav_step": STEP_BYTES_VELOCITY_QUAD,
                                 "frac": n_local * STEP_BYTES_VELOCITY_QUAD / (step_ms_no_imu * 1e-3) / 1e9 / peaks["hbm_gbs"]},
                "fp64": {"achieved_tflops_as_written_census": n_local * STEP_FLOP_VELOCITY_QUAD / (step_ms * 1e-3) / 1e12,
                         "peak_tflops_measured_dfma": fp64.value, "flop_per_uav_step_as_written": STEP_FLOP_VELOCITY_QUAD},
                "copy_gbs_measured_here": copy.value,
                "collision_pass": {"ms_avg_in_tick": tick_ms - step_ms, "share_of_tick": (tick_ms - step_ms) / tick_ms, "cell_m": info1["cell"],
                                   "neighbour_lists": info1["neighbour_lists"], "list_radius_m": info1["list_radius"], "skin_m": info1["skin"],
                                   "rebuild_fraction": (info1["rebuilds"] - info0["rebuilds"]) / passes, "ms_rebuild_pass_alone": coll_rebuild_ms,
                                   "ms_list_only_tick": list_tick_ms, "crowded_uavs_at_last_rebuild": info1["crowded_uavs"],
                                   "directed_pairs_last_tick": pairs_last}}
    if ex_flop:
        tf = n_local * ex_flop / (step_ms * 1e-3) / 1e12
        roofline["fp64"].update({"executed_flop_per_uav_step": ex_flop, "achieved_tflops_executed": tf,
                                 "frac_of_measured_dfma_peak": min(tf, roofline["fp64"]["achieved_tflops_as_written_census"]) / fp64.value})
    traffic_file = os.path.join(ROOT, "profiles", "step_kernel_traffic.json")
    if os.path.exists(traffic_file):
        with open(traffic_file) as f:
            roofline["traffic"] = json.load(f).get("dram_bytes_per_uav_step") * n_local  # ncu dram read+write per launch, scaled to this shard

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v1, _, _ = cpu_reference(65536, 2, 1, threads)
        ticks = int(max(3, min(60, 15.0 * v1 / N_UAVS)))
        v, _, desc = cpu_reference(N_UAVS, ticks, 2, threads)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc + "; " + port_vs_reference_sources()}
        try:
            vf, _, descf = cpu_reference(262144, max(3, ticks // 2), 1, threads, fast=True)
            cpu["fast_build"] = {"value": vf, "sample": descf}
        except Exception as e:  # no compiler on this host, or the build failed: the parity build above is the baseline
            cpu["fast_build"] = {"unavailable": str(e)[:200]}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": tick_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": cfg, "exchange": exchange, "clocks": clocks,
            "regime": f"mixed: timed after {args.fast_forward} untimed ticks of flight; value = median of {args.reps} blocks of {args.steps} ticks, each one mrsb_run call",
            "regimes": {"mixed": {"value": value, "ms_per_step": tick_ms, "blocks_ms": blocks, "best_block_value": N_UAVS * args.steps / (min(blocks) * 1e-3),
                                  "rebuild_fraction": (info1["rebuilds"] - info0["rebuilds"]) / passes, "directed_pairs_last_tick": pairs_last},
                        "fresh_grid": fresh, "l2_resident": resident},
            "state_checksum": {"x_u64_sum": f"{cs:016x}", "after_ticks": ticks_flown,
                               "note": "wrapping sum of the uint64 words of every UAV's position after the timed region: identical for every --gpus N"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(cmd_host.numel() * 8), "d2h_bytes_per_step": int(pos_host[0].numel() * 8),
                    "steps": n_e2e, "blocking_api_value": N_UAVS * min(n_e2e, 50) / e2e_blocking_s,
                    "commands_every_10th_tick_value": N_UAVS * n_e2e / e2e_10_s,
                    "commands_every_10th_tick_positions_of_every_4th_uav_value": N_UAVS * n_e2e / e2e_sub_s,
                    "h2d_gbs_achieved": cmd_host.numel() * 8 * n_e2e / e2e_s / 1e9, "d2h_gbs_achieved": pos_host[0].numel() * 8 * n_e2e / e2e_s / 1e9,
                    "note": "per rank, every tick, via the C ABI: VelocityHdgRate rows H2D from pinned memory (mrsb_set_input_async), one tick (mrsb_run), "
                            "positions D2H to pinned memory (mrsb_get_positions_async); upload of tick t+1 and download of tick t-1 overlap tick t on "
                            "separate streams (the tick is then as long as its PCIe upload: see h2d_gbs_achieved); commands_every_10th_tick_value = commands "
                            "uploaded on every 10th tick only (callback rate below tick rate), positions still downloaded every tick; "
                            "..._positions_of_every_4th_uav_value = the same with mrsb_set_position_subset(every 4th UAV): 6.3 MB down per tick; "
                            "blocking_api_value = mrsb_set_input + mrsb_get_state"},
            "gpu_launches": int(round(launches)), "roofline": roofline, "cpu_baseline": cpu, "secondary": secondary, "parity": parity}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--fast-forward", type=int, default=600, dest="fast_forward")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", dest="dump_outputs",
                    help="write what the timed path computed in its last tick as DIR/<name>.npy (one GPU only)")
    args = ap.parse_args()
    if args.dump_outputs and (args.gpus != 1 or args.impl != "b200"):
        ap.error("--dump-outputs needs --gpus 1 and --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
