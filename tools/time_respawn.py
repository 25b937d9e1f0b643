#!/usr/bin/env python
"""What an episode reset costs on the GPU (CUDA events on the handle's stream; card name and power limit read in the same run):
  1. mrsb_respawn_masked_device alone at 1 Mi UAVs, 1 % and 100 % of the mask set: time, and algorithmic bytes over time against
     the measured device-to-device copy bandwidth (mrsb_microbench_copy);
  2. the C3 loop (65,536 x500, VelocityHdg, K = 10) as an RL loop {masked respawn of p % -> mrsb_set_input_device for all ->
     make_step(0.01, 10)} for p = 0, 1, 100, beside the same loop without the respawn call, with the stepping kernel it ran;
  3. the bench workload (1 Mi x500, collisions, neighbour lists) through mrsb_run one tick at a time, in the same order
     {masked respawn of p % at their spawn points -> the bench's commands for all from the device -> one tick} for p = 0, 0.01 %
     and 1 %, beside the same ticks without the respawn call: tick time and rebuild fraction."""
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
# bytes the respawn of one UAV writes: st 18 + rpm 8 + pid 24 + cmd 12 + ff 13 + fext/mext/imu 9 + initz 1 doubles, flags 4,
# mode 1, packed position 24; and reads: xyz 24 + heading 8, parameter-set index 4, take-off flag 1
W_UAV = 8 * (18 + 8 + 24 + 12 + 13 + 9 + 1) + 4 + 1 + 24
R_UAV = 24 + 8 + 4 + 1


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def mask_of(n, p, seed):
    u = torch.rand(n, generator=torch.Generator(device=DEV).manual_seed(seed), device=DEV)
    return u < p


def timed(stream, fn, reps):
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record(stream)
    for r in range(reps):
        fn(r)
    e.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(e) * 1000.0 / reps  # us


def mask_kernel_alone(out):
    n = 1 << 20
    spawn, _ = workload(0, n)
    b = UavBatch([x500_world()], spawn_xyz=spawn, n=n)
    st = torch.cuda.ExternalStream(b.stream)
    xyz = torch.as_tensor(spawn, device=DEV)
    hdg = torch.zeros(n, dtype=torch.float64, device=DEV)
    copy = C.c_double(0.0)
    _lib.check(_lib.lib().mrsb_microbench_copy(0, C.byref(copy)))
    rows = {}
    for p in (0.01, 1.0):
        masks = [mask_of(n, p, 100 + k) for k in range(8)]
        torch.cuda.synchronize()
        for m in masks:  # warm-up
            b.respawn_masked_device(m.data_ptr(), xyz.data_ptr(), hdg.data_ptr())
        us = timed(st, lambda r: b.respawn_masked_device(masks[r % 8].data_ptr(), xyz.data_ptr(), hdg.data_ptr()), 200)
        hit = float(np.mean([int(m.sum()) for m in masks]))
        nbytes = n * 1 + hit * (W_UAV + R_UAV)  # the mask is read for every UAV
        rows[f"{p:.0%}"] = {"us": us, "respawned": hit, "algorithmic_bytes": nbytes, "GB_s": nbytes / us / 1e3, "of_copy_bw": nbytes / us / 1e3 / copy.value}
    out["mask_kernel_1Mi"] = {"copy_GB_s": copy.value, **rows}
    b.close()


def c3_loop(out):
    n, K = 65536, 10
    spawn, _ = workload(0, n)
    rng = np.random.default_rng(3)
    cmd = torch.as_tensor(np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n), rng.uniform(0.2, 1.5, n), rng.uniform(-3, 3, n)], axis=1), device=DEV)
    xyz = torch.as_tensor(spawn, device=DEV)
    hdg = torch.zeros(n, dtype=torch.float64, device=DEV)
    rows = {}
    for p in (None, 0.0, 0.01, 1.0):
        b = UavBatch([x500_world()], spawn_xyz=spawn, n=n)
        st = torch.cuda.ExternalStream(b.stream)
        masks = [mask_of(n, p or 0.0, 200 + k) for k in range(8)]
        torch.cuda.synchronize()

        def it(r):
            if p is not None:
                b.respawn_masked_device(masks[r % 8].data_ptr(), xyz.data_ptr(), hdg.data_ptr())
            b.set_input_device(VELOCITY_HDG_CMD, cmd.data_ptr(), 4)
            b.make_step(0.01, K)

        for r in range(20):
            it(r)
        us = timed(st, it, 300)
        rows["no respawn call" if p is None else f"{p:.0%}"] = {"us_per_iteration": us, "step_info": b.step_info()}
        b.close()
    out["c3_loop_65536_K10"] = rows


def bench_ticks(out):
    n = 1 << 20
    spawn, cmd = workload(0, n)
    xyz = torch.as_tensor(spawn, device=DEV)
    hdg = torch.zeros(n, dtype=torch.float64, device=DEV)
    cmd_dev = torch.as_tensor(cmd, device=DEV)
    rows = {}
    for p in (None, 0.0, 0.0001, 0.01):
        b = UavBatch([x500_world()], spawn_xyz=spawn, n=n)
        b.set_input(VELOCITY_HDG_RATE_CMD, cmd)
        b.set_collisions(True, False, 100.0)
        b.run(0.01, 300, with_collisions=True)  # into the steady state of the workload
        st = torch.cuda.ExternalStream(b.stream)
        masks = [mask_of(n, p or 0.0, 300 + k) for k in range(8)]
        torch.cuda.synchronize()

        def tick(r):
            if p is not None:
                b.respawn_masked_device(masks[r % 8].data_ptr(), xyz.data_ptr(), hdg.data_ptr())
            b.set_input_device(VELOCITY_HDG_RATE_CMD, cmd_dev.data_ptr(), 4)
            b.run(0.01, 1, with_collisions=True)

        i0 = b.collision_info()
        us = timed(st, tick, 400)
        i1 = b.collision_info()
        rows["no respawn call" if p is None else f"{p:.2%}"] = {"tick_us": us, "rebuild_fraction": (i1["rebuilds"] - i0["rebuilds"]) / max(1, i1["passes"] - i0["passes"])}
        b.close()
    out["bench_1Mi_ticks"] = rows


def main():
    out = {"card": card()}
    mask_kernel_alone(out)
    c3_loop(out)
    bench_ticks(out)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
