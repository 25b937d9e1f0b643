#!/usr/bin/env python
"""What mrsb_pack_neighbours_device costs on the GPU (CUDA events on the handle's stream after a warm-up; card name and power limit
read in the same run).  Two swarms:
  bench  1,048,576 x500 of bench.py (1024 x 1024 grid, 4 m pitch, VelocityHdgRate commands, collisions on), flown 600 ticks;
  C3     65,536 x500 of bench.py's C3 (256 x 256 grid at z = 10 m, random VelocityHdg commands), flown 100 launches of K = 10.
For radii 2, 5 and 10 m and k = 4, 8, 16: the time of one call (all three outputs), and, from a torch.profiler run of its own, the
split into table build (pack + count + scan + scatter) and query; the mean number of UAVs within the radius (the call's counts) and
the mean number of table records a UAV's query examines (its stencil's buckets, counted on the host from the same positions and
the same hash); algorithmic bytes (state rows 0-5 in, idx + rows + count out) over the call time, against the measured
device-to-device copy bandwidth (mrsb_microbench_copy)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import SEED, u01, workload, x500_world  # noqa: E402
from mrs_multirotor_simulator_b200 import VELOCITY_HDG_CMD, VELOCITY_HDG_RATE_CMD, UavBatch, _lib, airframe  # noqa: E402

DEV = torch.device("cuda:0")
RADII = (2.0, 5.0, 10.0)
KS = (4, 8, 16)
ROWS = 2  # stencil rows per axis of the table (collide.cu): cell = 2 * reach, 2 x 2 rows of 2 cells
TABLE_KERNELS = ("nb_pack_kernel", "count_kernel", "scan_kernel", "scatter_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def row_hash(cy, cz):
    """collide.cu row_hash, on uint32 arrays."""
    cy, cz = cy.astype(np.uint32), cz.astype(np.uint32)
    with np.errstate(over="ignore"):
        h = (cy * np.uint32(0x9E3779B1)) ^ (cz * np.uint32(0x85EBCA77) + np.uint32(0x165667B1))
        h ^= h >> np.uint32(15)
        h *= np.uint32(0x2C1B3C6D)
        h ^= h >> np.uint32(12)
    return h


def candidates_per_uav(x, radius):
    """Mean number of records in the stencil of a UAV (what the query walks), from the table layout of api.cu / collide.cu."""
    n = len(x)
    bits = 10
    while 2 * (1 << bits) < 3 * n and bits < 30:
        bits += 1
    mask = np.uint32((1 << bits) - 1)
    reach = radius * (1.0 + 2.0 ** -20)
    inv_cell = 1.0 / (2.0 * reach / (ROWS - 1))
    cell = np.floor(x * inv_cell).astype(np.int64).astype(np.int32)
    with np.errstate(over="ignore"):
        b = (row_hash(cell[:, 1], cell[:, 2]) + cell[:, 0].astype(np.uint32)) & mask
    occ = np.bincount(b, minlength=int(mask) + 1 + ROWS)
    occ[int(mask) + 1:int(mask) + ROWS] = occ[:ROWS - 1]  # mirror buckets
    c0 = np.floor((x - reach) * inv_cell).astype(np.int64).astype(np.int32)
    total = np.zeros(n, dtype=np.int64)
    for a in range(ROWS * ROWS):
        with np.errstate(over="ignore"):
            b0 = (row_hash(c0[:, 1] + a % ROWS, c0[:, 2] + a // ROWS) + c0[:, 0].astype(np.uint32)) & mask
        for t in range(ROWS):
            total += occ[b0.astype(np.int64) + t]
    return float(total.mean())


def bench_swarm():
    n = 1 << 20
    spawn, cmd = workload(0, n)
    b = UavBatch([x500_world()], spawn_xyz=spawn, n=n)
    b.set_input(VELOCITY_HDG_RATE_CMD, cmd)
    b.set_collisions(True, False, 100.0)
    b.run(0.01, 600, with_collisions=True)
    return b


def c3_swarm():
    n = 65536
    k = np.arange(n)
    spawn = np.stack([4.0 * (k % 256), 4.0 * (k // 256), np.full(n, 10.0)], axis=1)
    cmd = np.ascontiguousarray(np.stack([-2 + 4 * u01(SEED, 1, k), -2 + 4 * u01(SEED, 2, k), -2 + 4 * u01(SEED, 3, k),
                                         -np.pi + 2 * np.pi * u01(SEED, 4, k)], axis=1))
    b = UavBatch([airframe("x500")], spawn_xyz=spawn, n=n)
    b.set_input(VELOCITY_HDG_CMD, cmd)
    for _ in range(100):
        b.make_step(0.01, 10)
    return b


def timed(stream, fn, reps):
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record(stream)
    for _ in range(reps):
        fn()
    e.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(e) * 1000.0 / reps  # us


def kernel_split(fn, reps):
    """Per-call device time of the table kernels and of the query kernel, from a profiler run of its own."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    table = query = 0.0
    for ev in prof.key_averages():
        t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if "nb_query_kernel" in ev.key:
            query += t
        elif any(k in ev.key for k in TABLE_KERNELS):
            table += t
    return table / reps, query / reps


def measure(name, b, copy_gbs, out):
    n = b.n
    x = b.get_state(fields=("x",))["x"]
    st = torch.cuda.ExternalStream(b.stream)
    idx = torch.empty((n, 16), dtype=torch.int32, device=DEV)
    rows = torch.empty((n, 96), dtype=torch.float64, device=DEV)
    cnt = torch.empty(n, dtype=torch.int32, device=DEV)
    res = {}
    for r in RADII:
        cand = candidates_per_uav(x, r)
        for k in KS:
            def call():
                b.pack_neighbours_device(r, k, idx.data_ptr(), rows.data_ptr(), cnt.data_ptr())

            for _ in range(5):
                call()
            us = timed(st, call, 50)
            table_us, query_us = kernel_split(call, 10)
            within = float(cnt.double().mean())
            nbytes = n * (48 + 4 * k + 48 * k + 4)
            res[f"r={r:g} k={k}"] = {"call_us": us, "table_us": table_us, "query_us": query_us, "mean_within_radius": within,
                                     "mean_candidates": cand, "algorithmic_bytes": nbytes, "GB_s": nbytes / us / 1e3,
                                     "of_copy_bw": nbytes / us / 1e3 / copy_gbs}
    out[name] = {"n": n, **res}


def main():
    copy = C.c_double(0.0)
    _lib.check(_lib.lib().mrsb_microbench_copy(0, C.byref(copy)))
    out = {"card": card(), "copy_GB_s": copy.value}
    for name, make in (("bench_1Mi_600_ticks", bench_swarm), ("c3_65536", c3_swarm)):
        b = make()
        measure(name, b, copy.value, out)
        b.close()
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
