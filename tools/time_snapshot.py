#!/usr/bin/env python
"""What saving and restoring snapshots costs on the GPU (CUDA events on the handle's stream; card name and power limit read in the
same run):
  1. on the bench swarm (1 Mi x500 after 300 ticks of the bench workload): mrsb_snapshot_save, the full host restore (every UAV
     its own record), and the device restore with 1 % and 100 % of the UAVs selected, each with its own record ("identity") and
     with a random record ("random"); time, and algorithmic bytes over time against the device-to-device copy bandwidth
     measured in the same run (mrsb_microbench_copy);
  2. the C3 loop (65,536 x500, VelocityHdg, K = 10) as an RL loop {reset -> mrsb_set_input_device for all -> make_step(0.01, 10)}
     with the reset a device restore of 1 % / 100 % of the UAVs from their own records, beside the same loop with
     mrsb_respawn_masked_device of the same UAVs, with the stepping kernel each ran.
The snapshot (743 MB at 1 Mi UAVs) and the state it is copied to are larger than the 126 MB L2: no flush between calls."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import workload, x500_world  # noqa: E402
from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD, VELOCITY_HDG_RATE_CMD, UavBatch, _lib  # noqa: E402

DEV = torch.device("cuda:0")
RECORD = 88 * 8 + 4 + 1  # bytes of one UAV's snapshot record
GPOS = 24  # the packed position a restore also writes
SRC = 4  # the src word the device restore reads for every UAV


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def timed(stream, fn, reps):
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record(stream)
    for r in range(reps):
        fn(r)
    e.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(e) * 1000.0 / reps  # us


def srcs(n, p, kind, seed):
    """Eight device src arrays: a fraction p of the UAVs selected (record = own index, or a random one), -1 elsewhere."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    out = []
    for _ in range(8):
        sel = torch.rand(n, generator=g, device=DEV) < p
        rec = torch.arange(n, device=DEV, dtype=torch.int32) if kind == "identity" else torch.randint(0, n, (n,), generator=g, device=DEV,
                                                                                                            dtype=torch.int32)
        out.append(torch.where(sel, rec, torch.full_like(rec, -1)))
    return out


def row(us, nbytes, copy):
    return {"us": us, "algorithmic_bytes": nbytes, "GB_s": nbytes / us / 1e3, "of_copy_bw": nbytes / us / 1e3 / copy}


def bench_swarm(out):
    n = 1 << 20
    spawn, cmd = workload(0, n)
    b = UavBatch([x500_world()], spawn_xyz=spawn, n=n)
    b.set_input(VELOCITY_HDG_RATE_CMD, cmd)
    b.set_collisions(True, False, 100.0)
    b.run(0.01, 300, with_collisions=True)
    st = torch.cuda.ExternalStream(b.stream)
    copy = C.c_double(0.0)
    _lib.check(_lib.lib().mrsb_microbench_copy(0, C.byref(copy)))
    s = b.snapshot()
    s.save()
    rows = {"copy_GB_s": copy.value}
    for _ in range(5):
        s.save()
    rows["save"] = row(timed(st, lambda r: s.save(), 100), n * 2 * RECORD, copy.value)
    for _ in range(5):
        s.restore()
    rows["restore_all_host"] = row(timed(st, lambda r: s.restore(), 100), n * (2 * RECORD + GPOS), copy.value)
    for p in (0.01, 1.0):
        for kind in ("identity", "random"):
            ss = srcs(n, p, kind, 7)
            hit = float(np.mean([int((x >= 0).sum()) for x in ss]))
            torch.cuda.synchronize()
            for x in ss:
                s.restore_device(x.data_ptr())
            us = timed(st, lambda r: s.restore_device(ss[r % 8].data_ptr()), 100)
            rows[f"restore_device_{p:.0%}_{kind}"] = {"restored": hit, **row(us, n * SRC + hit * (2 * RECORD + GPOS), copy.value)}
    out["bench_swarm_1Mi"] = rows
    s.free()
    b.close()


def c3_loop(out):
    n, K = 65536, 10
    spawn, _ = workload(0, n)
    rng = np.random.default_rng(3)
    cmd = torch.as_tensor(np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n), rng.uniform(0.2, 1.5, n), rng.uniform(-3, 3, n)], axis=1), device=DEV)
    xyz = torch.as_tensor(spawn, device=DEV)
    hdg = torch.zeros(n, dtype=torch.float64, device=DEV)
    rows = {}
    for p in (0.01, 1.0):
        for how in ("restore_device", "respawn_masked_device"):
            b = UavBatch([x500_world()], spawn_xyz=spawn, n=n)
            st = torch.cuda.ExternalStream(b.stream)
            b.set_input_device(VELOCITY_HDG_CMD, cmd.data_ptr(), 4)
            b.make_step(0.01, K)
            s = b.snapshot()
            s.save()
            ss = srcs(n, p, "identity", 11)
            masks = [x >= 0 for x in ss]
            torch.cuda.synchronize()

            def it(r):
                if how == "restore_device":
                    s.restore_device(ss[r % 8].data_ptr())
                else:
                    b.respawn_masked_device(masks[r % 8].data_ptr(), xyz.data_ptr(), hdg.data_ptr())
                b.set_input_device(VELOCITY_HDG_CMD, cmd.data_ptr(), 4)
                b.make_step(0.01, K)

            for r in range(20):
                it(r)
            us = timed(st, it, 300)
            rows[f"{how}_{p:.0%}"] = {"us_per_iteration": us, "step_info": b.step_info()}
            s.free()
            b.close()
    out["c3_loop_65536_K10"] = rows


def main():
    out = {"card": card()}
    bench_swarm(out)
    c3_loop(out)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
