"""A handle gives back all the device memory it took: create, touch every buffer that grows on demand, destroy, many times over,
and the free memory of the device does not drift.  Also for a create that fails after it has allocated.

Free memory is read with torch.cuda.mem_get_info, so other work on the same GPU disturbs it: run this file alone there."""
import numpy as np
import pytest

from helpers import grid_spawn
from oracle import binding as O

pytestmark = pytest.mark.gpu

N = 256 * 1024  # UAVs per handle: a footprint of a few hundred MB, far above the noise of the free-memory reading
CYCLES = 20


def af(name, **kw):
    from mrs_multirotor_simulator_b200 import airframe

    return airframe(name, **kw)


def free_bytes():
    import torch

    torch.cuda.synchronize()
    return torch.cuda.mem_get_info(0)[0]


def make(mixed):
    from mrs_multirotor_simulator_b200 import UavBatch

    if mixed:
        tou = (np.arange(N) % 3).astype(np.int32)  # three airframes: a bucketed handle
        return UavBatch([af("x500"), af("f550"), af("t650")], type_of_uav=tou, spawn_xyz=grid_spawn(N, z=5.0), n=N)
    return UavBatch([af("x500")], spawn_xyz=grid_spawn(N, z=5.0), n=N)


def touch_every_grow_path(b, pinned):
    cmd, pos, sub_pos = pinned
    b.get_state()  # staging buffer: the widest full-swarm rows
    b.get_odometry()
    idx = np.arange(0, N, 3, dtype=np.int32)  # index list
    b.set_input(O.POSITION_CMD, np.tile([1.0, 2.0, 3.0, 0.5], (len(idx), 1)), idx=idx)
    b.set_mass(1.5 + 0.01 * np.arange(40), idx=np.arange(40, dtype=np.int32))  # 40 distinct values: a larger parameter table
    b.set_input_async(O.POSITION_CMD, cmd.data_ptr(), 4)  # upload and download pipeline
    b.get_positions_async(pos.data_ptr())
    b.set_position_subset(np.arange(0, N, 7, dtype=np.int32))
    b.get_positions_async(sub_pos.data_ptr())
    b.set_pair_capacity(8 * N)  # above the default of 4 per UAV
    b.sync()


def pinned_buffers():
    import torch

    cmd = torch.from_numpy(np.tile([1.0, 2.0, 3.0, 0.5], (N, 1))).pin_memory()
    pos = torch.zeros((N, 3), dtype=torch.float64).pin_memory()
    sub_pos = torch.zeros((len(range(0, N, 7)), 3), dtype=torch.float64).pin_memory()
    return cmd, pos, sub_pos


@pytest.mark.parametrize("mixed", [False, True], ids=["uniform", "bucketed"])
def test_destroy_frees_everything_a_handle_grew(mixed):
    pinned = pinned_buffers()
    before = free_bytes()
    b = make(mixed)  # the first cycle also loads the kernels: the baseline is taken after it
    touch_every_grow_path(b, pinned)
    footprint = before - free_bytes()
    b.close()
    baseline = free_bytes()
    for _ in range(CYCLES):
        b = make(mixed)
        touch_every_grow_path(b, pinned)
        b.close()
    drop = baseline - free_bytes()
    assert footprint > 0
    assert drop < footprint / 2, f"{drop / 2**20:.1f} MiB less free memory after {CYCLES} handles of {footprint / 2**20:.1f} MiB"


def test_failed_create_frees_what_it_allocated():
    """type_of_uav of a remote UAV is only checked once the handle's device arrays exist."""
    from mrs_multirotor_simulator_b200 import UavBatch
    from mrs_multirotor_simulator_b200._lib import MrsbError

    types = [af("x500"), af("f550")]
    spawn = grid_spawn(N, z=5.0)
    good = (np.arange(2 * N) % 2).astype(np.int32)
    bad = good.copy()
    bad[N + 5] = 7  # remote half, outside 0..1
    before = free_bytes()
    b = UavBatch(types, type_of_uav=good, spawn_xyz=spawn, n=N, n_global=2 * N)
    footprint = before - free_bytes()
    b.close()
    baseline = free_bytes()
    for _ in range(CYCLES):
        with pytest.raises(MrsbError) as e:
            UavBatch(types, type_of_uav=bad, spawn_xyz=spawn, n=N, n_global=2 * N)
        assert e.value.code == -1  # MRSB_ERR_INVALID
        assert "type_of_uav" in str(e.value)
    drop = baseline - free_bytes()
    assert footprint > 0
    assert drop < footprint / 2, f"{drop / 2**20:.1f} MiB less free memory after {CYCLES} failed creates (handle: {footprint / 2**20:.1f} MiB)"
