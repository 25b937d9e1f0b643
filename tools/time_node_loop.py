#!/usr/bin/env python
"""What a multi-UAV node's tick costs end to end through the pipelined calls (card name and power limit read in the same run).

The bench swarm (1 Mi x500, bench.py's workload) is flown untimed for 300 ticks.  Every regime then runs blocks of ticks, each block
ending in mrsb_sync; the median block gives the time per tick.  Per tick, through the C ABI:
  whole_batch_async     VelocityHdgRate rows of every UAV (mrsb_set_input_async), mrsb_run, positions of every UAV
                        (mrsb_get_positions_async) — bench.py's e2e path, the reference point;
  rows_1pct / rows_10pct  VelocityHdgRate rows of 1 % / 10 % of the UAVs (mrsb_set_input_rows_async), run, positions;
  rows_10pct_mixed      10 % rows in five modes (the stepping kernel runs its per-UAV-mode path), run, positions;
  rows_10pct_obs_all / rows_10pct_obs_every4th  10 % VelocityHdgRate rows, run, odometry | IMU | range rows of every UAV / of every
                        4th UAV (mrsb_get_observations_async).
Each regime draws 4 sets of rows (UAVs chosen without repetition, in random order) and cycles through them; a regime with
VelocityHdgRate rows starts with one whole-batch call, so that the batch is single-mode.  Reported per regime: time per tick, bytes
up and down per tick and those bytes over the tick time, host time inside the row call (it validates every row on the host), and
the stepping kernel of the last tick.  The claim and apply kernels alone are timed with CUDA events at 10 k and 1 Mi rows, with the
stream busy with ticks while the rows upload, so that the events hold the two kernels and nothing else.  Last, a twin handle flown
the same 300 ticks takes 20 ticks of mixed rows through the blocking calls; the states must be equal bit for bit.
Writes the JSON to stdout and, with --out, to that file."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import workload, x500_world  # noqa: E402
from mrs_multirotor_simulator_b200 import (ACCELERATION_HDG_CMD, ACCELERATION_HDG_RATE_CMD, POSITION_CMD, VELOCITY_HDG_CMD,  # noqa: E402
                                           VELOCITY_HDG_RATE_CMD, UavBatch, _lib)

N = 1 << 20
DT = 0.01
MIXED = [VELOCITY_HDG_RATE_CMD, VELOCITY_HDG_CMD, ACCELERATION_HDG_RATE_CMD, ACCELERATION_HDG_CMD, POSITION_CMD]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def pinned(a):
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


class Rows:
    """One set of command rows in pinned memory: `count` UAVs without repetition, in random order, rows of 4 doubles."""

    def __init__(self, rng, spawn, cmd, count, modes):
        idx = rng.permutation(N)[:count].astype(np.int32)
        mode = rng.choice(modes, count).astype(np.int32)
        rows = cmd[idx].copy()
        pos = mode == POSITION_CMD  # a waypoint near the spawn point, not across the swarm
        rows[pos, :3] = spawn[idx[pos]] + np.array([1.0, -1.0, 3.0])
        self.n, self.idx, self.modes, self.rows = count, pinned(idx), pinned(mode), pinned(rows)
        self.host = (idx, mode, rows)

    def send(self, b):
        _lib.check(b._L.mrsb_set_input_rows_async(b.h, self.n, C.c_void_p(self.idx.data_ptr()), C.c_void_p(self.modes.data_ptr()),
                                                  C.c_void_p(self.rows.data_ptr()), 4))


def send_blocking(b, r):
    """The same rows through mrsb_set_input, one call per mode (the UAVs of one set are distinct)."""
    idx, mode, rows = r.host
    for m in np.unique(mode):
        i = np.ascontiguousarray(idx[mode == m])
        p = np.ascontiguousarray(rows[mode == m])
        _lib.check(b._L.mrsb_set_input(b.h, int(m), len(i), i.ctypes.data_as(C.c_void_p), p.ctypes.data_as(C.c_void_p), 4))


def regime(b, whole_cmd, kind, rows=None, obs_every=0, ticks=50, blocks=7):
    L = b._L
    m = N if obs_every <= 1 else len(range(0, N, obs_every))
    b.set_position_subset(np.arange(0, N, obs_every, dtype=np.int32) if obs_every > 1 else None)
    pos = [torch.empty((m, 3), dtype=torch.float64).pin_memory() for _ in range(2)]
    obs = [torch.empty((m, 17), dtype=torch.float64).pin_memory() for _ in range(2)] if obs_every else None
    if kind != "whole" and (rows is None or all(int(x) == VELOCITY_HDG_RATE_CMD for x in rows[0].host[1])):
        _lib.check(L.mrsb_set_input_async(b.h, VELOCITY_HDG_RATE_CMD, C.c_void_p(whole_cmd.data_ptr()), 4))  # single-mode batch
    host_s = []

    def tick(t):
        if kind == "whole":
            _lib.check(L.mrsb_set_input_async(b.h, VELOCITY_HDG_RATE_CMD, C.c_void_p(whole_cmd.data_ptr()), 4))
        else:
            h0 = time.perf_counter()
            rows[t % len(rows)].send(b)
            host_s.append(time.perf_counter() - h0)
        _lib.check(L.mrsb_run(b.h, DT, 1, 1, 1))
        if obs is None:
            _lib.check(L.mrsb_get_positions_async(b.h, C.c_void_p(pos[t & 1].data_ptr())))
        else:
            _lib.check(L.mrsb_get_observations_async(b.h, C.c_void_p(obs[t & 1].data_ptr())))

    for t in range(10):
        tick(t)
    b.sync()
    ms = []
    for _ in range(blocks):
        t0 = time.perf_counter()
        for t in range(ticks):
            tick(t)
        b.sync()
        ms.append((time.perf_counter() - t0) * 1e3 / ticks)
    tick_ms = float(np.median(ms))
    up = N * 32 if kind == "whole" else rows[0].n * (4 + 4 + 32)
    down = m * (17 * 8 if obs is not None else 24)
    out = {"ms_per_tick": round(tick_ms, 4), "ms_per_tick_blocks": [round(x, 4) for x in ms], "G_uav_steps_per_s": round(N / tick_ms / 1e6, 3),
           "rows_per_tick": N if kind == "whole" else rows[0].n, "h2d_bytes_per_tick": up, "d2h_bytes_per_tick": down,
           "h2d_GB_s_over_tick": round(up / tick_ms / 1e6, 2), "d2h_GB_s_over_tick": round(down / tick_ms / 1e6, 2),
           "step_info": b.step_info()}
    if host_s:
        out["host_us_in_row_call_median"] = round(float(np.median(host_s)) * 1e6, 1)
    b.set_position_subset(None)
    return out


def kernel_times(b, spawn, cmd, rng, reps=20):
    """claim + apply of one row call, by CUDA events on the handle's stream; five ticks ahead of each call keep the stream busy
    while the rows upload, so the stream finds them on the device and the events hold the two kernels only."""
    st = torch.cuda.ExternalStream(b.stream)
    out = {}
    for count in (10_000, N):
        r = Rows(rng, spawn, cmd, count, [VELOCITY_HDG_RATE_CMD])
        r.send(b)
        b.sync()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for e0, e1 in ev:
            b.run(DT, 5)
            e0.record(st)
            r.send(b)
            e1.record(st)
        b.sync()
        us = [e0.elapsed_time(e1) * 1e3 for e0, e1 in ev]
        out[str(count)] = {"claim_plus_apply_us_median": round(float(np.median(us)), 2), "us_min": round(min(us), 2)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    args = ap.parse_args()
    out = {"card": card(), "n_uavs": N, "warm_ticks": 300}
    spawn, cmd = workload(0, N)
    rng = np.random.default_rng(5)
    b = UavBatch([x500_world()], spawn_xyz=spawn, n=N)
    twin = UavBatch([x500_world()], spawn_xyz=spawn, n=N)
    for s in (b, twin):
        s.set_input(VELOCITY_HDG_RATE_CMD, cmd)
        s.set_collisions(True, False, 100.0)
        s.run(DT, 300)
    # equality with the blocking calls: 20 ticks of 10 % mixed rows
    sets = [Rows(rng, spawn, cmd, N // 10, MIXED) for _ in range(4)]
    for t in range(20):
        sets[t % 4].send(b)
        send_blocking(twin, sets[t % 4])
        for s in (b, twin):
            s.run(DT, 1)
    b.sync()
    fa, fb = b.get_full_state(), twin.get_full_state()
    out["equal_to_blocking_twin"] = bool(all(np.array_equal(fa[k], fb[k]) for k in fa)) and bool(np.array_equal(b.get_input_mode(), twin.get_input_mode()))
    twin.close()
    whole = pinned(cmd)
    vhr = {p: [Rows(rng, spawn, cmd, int(N * p), [VELOCITY_HDG_RATE_CMD]) for _ in range(4)] for p in (0.01, 0.1)}
    R = {}
    R["whole_batch_async"] = regime(b, whole, "whole")
    R["rows_1pct"] = regime(b, whole, "rows", vhr[0.01])
    R["rows_10pct"] = regime(b, whole, "rows", vhr[0.1])
    R["rows_10pct_mixed"] = regime(b, whole, "rows", sets)
    R["rows_10pct_obs_all"] = regime(b, whole, "rows", vhr[0.1], obs_every=1)
    R["rows_10pct_obs_every4th"] = regime(b, whole, "rows", vhr[0.1], obs_every=4)
    out["regimes"] = R
    out["row_kernels"] = kernel_times(b, spawn, cmd, rng)
    out["note"] = ("ms_per_tick: median of 7 blocks of 50 ticks, each ending in mrsb_sync, host clock; *_GB_s_over_tick: bytes per tick over "
                   "the whole tick time (not a copy rate); rows of 4 doubles + int32 index + int32 mode; no L2 flush (the state is 1.5 GB)")
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
