"""Host side of a batch (batch.cu): what agarcl_batch_create refuses, batches on two devices of one process, and the kernels a
step launches."""
import re

import numpy as np
import pytest

from agarcl_b200 import make_cfg

pytestmark = pytest.mark.gpu


def test_too_much_shared_memory_is_refused():
    """22000 pellets need 246432 B of shared memory per instance (ag::make_smem_offsets), more than an SM has"""
    from agarcl_b200._lib import AgarclError
    from agarcl_b200.batch import Batch
    with pytest.raises(AgarclError, match="shared memory") as err:
        Batch(make_cfg(n_instances=2, num_pellets=22000))
    assert int(re.search(r"needs (\d+) B", str(err.value)).group(1)) == 246432


def test_batches_on_two_devices_of_one_process():
    """k_step and k_ram are set up on each device a batch is created on: the second device's batch steps like the first's"""
    import torch
    from agarcl_b200.batch import Batch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    N = 24
    kw = dict(n_instances=N, ram_obs=1, instance_base=5, num_bots=6, arena_size=300, num_pellets=300, num_viruses=4)
    rng = np.random.default_rng(4)
    actions = [(rng.uniform(-1, 1, size=(N, 2)).astype(np.float32), rng.integers(0, 3, size=N).astype(np.int32)) for _ in range(20)]
    outs = []
    for device in (0, 1):
        b = Batch(make_cfg(device=device, **kw))
        b.seed(77)
        b.reset()
        for dxdy, act in actions:
            b.set_actions(dxdy, act)
            b.step()
        torch.cuda.synchronize(device)
        outs.append((b.obs_tensor().cpu(), b.rewards_tensor().cpu(), b.ram_tensor().cpu(), [b.download_state(i).blob for i in range(N)]))
        b.close()
    (o0, r0, m0, s0), (o1, r1, m1, s1) = outs
    assert torch.equal(o0, o1) and torch.equal(r0, r1) and torch.equal(m0, m1)
    assert all(np.array_equal(a, b) for a, b in zip(s0, s1))


# kernels per step of configurations of gpu_parity_lib.CASES: k_step + k_order, + k_ram with ram_obs; two frames: four
# one-tick k_step launches, k_obs for each of the last two ticks and the closing k_step; strict_reference: k_obs renders the
# frame (ticks_per_step = 1)
LAUNCHES = {"mode9_deaths_and_limit": 2, "configs1_two_agents": 2, "int16": 2, "two_frames": 7, "strict_reference": 2,
            "ram_obs1": 3, "ram_obs2": 3, "mt19937_ring_wraps": 2}


@pytest.mark.parametrize("name", list(LAUNCHES))
def test_launches_per_step(name):
    from agarcl_b200.batch import Batch
    from gpu_parity_lib import CASES
    N = 8
    b = Batch(make_cfg(n_instances=N, **CASES[name][0]))
    b.seed(3)
    b.reset()
    b.set_actions(np.zeros((N * b.A, 2), np.float32), np.zeros(N * b.A, np.int32))
    b.step()
    assert b.launches_per_step() == LAUNCHES[name]
    b.close()
