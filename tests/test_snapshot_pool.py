"""CPU: the size of a snapshot slot (include/agarcl_b200.h, agarcl_snapshot_slot_bytes) follows the documented layout, needs no
device, and k_snapshot compiles for sm_100a without spills."""
import os
import re
import subprocess
import sys
import tempfile

import pytest

from _helpers import ROOT
from agarcl_b200 import OBS_I16, make_cfg, snapshot_slot_bytes
from agarcl_b200._abi import RAM_RECORD
from agarcl_b200._lib import make_layout


def _align(v, a):
    return (v + a - 1) // a * a


def documented_slot_bytes(cfg):
    """header 64 B | blob | episode record | ram records (ram_obs) | observation images (num_frames > 1, grid) | pad to 128"""
    L = make_layout(cfg)
    esz = 2 if cfg.obs_dtype == OBS_I16 else 4
    ep = _align(8 + 8 * L.A, 16)
    ram = L.P * 4 * RAM_RECORD if cfg.ram_obs else 0
    obs = 0
    if cfg.num_frames > 1 and cfg.ram_obs != 2:
        obs = _align(L.A * cfg.num_frames * L.obs_channels * cfg.grid_size * cfg.grid_size * esz, 16)
    return _align(64 + L.stride + ep + ram + obs, 128)


CASES = [dict(), dict(num_agents=2), dict(num_agents=5, num_bots=10), dict(ram_obs=1), dict(ram_obs=2, num_agents=3),
         dict(num_frames=3), dict(num_frames=3, grid_size=33, obs_dtype=OBS_I16, num_agents=2), dict(num_frames=3, ram_obs=2),
         dict(num_frames=2, ram_obs=1, observe_others=False), dict(obs_dtype=OBS_I16), dict(mode_number=9, num_bots=1, arena_size=200)]


@pytest.mark.parametrize("kw", CASES)
def test_slot_bytes_follow_the_documented_layout(kw):
    cfg = make_cfg(**kw)
    n = snapshot_slot_bytes(cfg)
    assert n == documented_slot_bytes(cfg)
    assert n % 128 == 0
    # what a batch size, a device, a shard or a replay capacity do not change
    assert snapshot_slot_bytes(make_cfg(n_instances=77, device=3, instance_base=1000, **kw)) == n


def test_one_frame_observation_is_not_stored():
    base = snapshot_slot_bytes(make_cfg())
    assert base == snapshot_slot_bytes(make_cfg(grid_size=64))  # re-rendered on restore, not stored
    assert snapshot_slot_bytes(make_cfg(num_frames=2)) - base >= 2 * 8 * 128 * 128 * 4
    assert base < 64 * 1024  # about 57 KB at configs[1]


def test_invalid_config_is_rejected():
    from agarcl_b200._lib import AgarclError
    with pytest.raises(AgarclError, match="mode"):
        snapshot_slot_bytes(make_cfg(mode_number=11))


def test_slot_bytes_need_no_device():
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from agarcl_b200 import make_cfg, snapshot_slot_bytes\n"
            "print(snapshot_slot_bytes(make_cfg(num_frames=2, ram_obs=1)))\n") % ROOT
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, check=True).stdout
    assert int(out) == documented_slot_bytes(make_cfg(num_frames=2, ram_obs=1))


def test_k_snapshot_has_no_spills():
    from agarcl_b200 import build
    flags = [f for f in build.NVCC_FLAGS if f != "-shared"]
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, "snapshot_kernel.cu"),
                                             "-o", os.path.join(d, "snapshot_kernel.o")], capture_output=True, text=True, check=True)
    text = r.stdout + r.stderr
    blocks = re.findall(r"Function properties for (\S*k_snapshot\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                        r"(\d+) bytes spill loads", text)
    assert len(blocks) == 2, text  # the save and the restore direction
    for name, stack, st, ld in blocks:
        assert (int(stack), int(st), int(ld)) == (0, 0, 0), (name, stack, st, ld)
