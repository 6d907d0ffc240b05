"""CPU: the layout of a mixed-task batch (cfg.task_modes, include/agarcl_b200.h): players and pellet capacity of a set of modes,
the refusals, the mode rules shared by the host and the kernels, and a layout without tasks exactly as before."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from _helpers import ROOT
from agarcl_b200 import make_cfg, snapshot_slot_bytes
from agarcl_b200._abi import task_bits
from agarcl_b200._lib import AgarclError, make_layout

# the ten AgarCL mini-games (bench/tasks_configs): arena 350, 500 pellets, no viruses
MINI = dict(arena_size=350, num_pellets=500, num_viruses=0, num_bots=0)


def set_mode_table(mode):
    """Engine::set_mode (Engine.hpp:367-416) and the bot roster of BaseEnvironment::reset, restated independently"""
    base = {5: 2, 6: 4}.get(mode, 4 if mode >= 7 else mode)
    return dict(mass_decay=int(base in (0, 2, 4)), squared_pellets=int(base in (1, 2)), regen=int(base in (0, 3, 4)),
                agent_mass=1000 if mode in (5, 6) else 25)


def bots_of(mode, num_bots):
    return num_bots if mode == 0 else (1 if mode > 6 else 0)


@pytest.mark.parametrize("mode", range(11))
def test_mode_rules_reproduce_the_flags_and_roster(mode):
    L = make_layout(make_cfg(mode_number=mode, num_agents=2, num_bots=6))
    for k, v in set_mode_table(mode).items():
        assert getattr(L, k) == v, (mode, k)
    assert L.P == 2 + bots_of(mode, 6)
    want = [-1, -1] + ([0, 1, 2, 3, 0, 0] if mode == 0 else [mode - 7] if mode > 6 else [])
    assert list(L.bot_type)[:L.P] == want


def test_layout_without_tasks_is_byte_identical_to_before():
    """tests/golden/layouts/no_tasks.npz: agarcl_layout bytes the library made before task_modes existed (all 11 modes, four
    configurations each)"""
    g = np.load(os.path.join(ROOT, "tests", "golden", "layouts", "no_tasks.npz"))
    keys = [str(k) for k in g["keys"]]
    assert len(g["layout"]) == 44
    for row, blob in zip(g["cfg"], g["layout"]):
        kw = {k: int(v) for k, v in zip(keys, row) if v != -1}
        L = make_layout(make_cfg(**kw))
        assert np.frombuffer(bytes(L), np.uint8).tobytes() == blob.tobytes(), kw


@pytest.mark.parametrize("modes", [(1, 2, 3, 4, 5, 6, 7, 8, 9, 10), (3, 4), (1, 3), (7, 8, 9, 10), (3, 9), (2,)])
def test_players_and_pellet_capacity_of_a_set(modes):
    for A in (1, 3):
        cfg = make_cfg(num_agents=A, mode_number=modes[0], task_modes=task_bits(modes), **MINI)
        L = make_layout(cfg)
        assert L.P == A + max(bots_of(m, 0) for m in modes)
        squared = any(set_mode_table(m)["squared_pellets"] for m in modes)
        assert L.cap_pellets == (700 if squared else 500)  # 4 * (350 // 2) for the squared-pellet modes
        # the mode flags and bot types stay mode_number's
        alone = make_layout(make_cfg(num_agents=A, mode_number=modes[0], **MINI))
        for k in ("mass_decay", "squared_pellets", "regen", "agent_mass"):
            assert getattr(L, k) == getattr(alone, k)
        # the slot: header + blob of this layout + episode record (+ nothing else here), and the task changes the fingerprint only
        assert snapshot_slot_bytes(cfg) == (64 + L.stride + (8 + 8 * A + 15) // 16 * 16 + 127) // 128 * 128


def test_mode_zero_shares_a_batch_with_modes_of_its_bot_count():
    L = make_layout(make_cfg(mode_number=0, task_modes=task_bits([0, 7, 8]), **dict(MINI, num_bots=1)))
    assert L.P == 2
    L = make_layout(make_cfg(mode_number=3, task_modes=task_bits([0, 1, 3]), **MINI))
    assert L.P == 1


@pytest.mark.parametrize("kw, msg", [
    (dict(task_modes=task_bits([1, 2]), strict_reference=True), "strict_reference"),
    (dict(task_modes=1 << 11), "outside 0..10"),
    (dict(task_modes=-1), "outside 0..10"),
    (dict(task_modes=task_bits([2, 3])), "must contain mode_number 1"),
    (dict(task_modes=task_bits([0, 1, 7]), mode_number=0), "mode 0 .* cannot share a batch with mode 7"),
    (dict(task_modes=task_bits([0, 1]), mode_number=1, num_bots=2), "mode 0 .* cannot share a batch with mode 1"),
])
def test_refusals_name_the_reason(kw, msg):
    cfg = make_cfg(**dict(dict(MINI, mode_number=1), **kw))
    with pytest.raises(AgarclError, match=msg):
        make_layout(cfg)


def libstdcxx_order(P):
    """the order unordered_map<unsigned short, int> iterates keys 0..P-1 in (agarcl_make_layout of a batch of P players)"""
    return list(make_layout(make_cfg(num_agents=P, num_bots=0, mode_number=1)).order)[:P]


def test_order_check_matches_the_batch_of_each_mode_alone():
    """every accepted set: the batch's order restricted to players < P_m is the order of mode m alone; a refused set is one where
    it is not.  With one agent (P <= 2) it always holds."""
    for A in range(1, 40):
        full, alone = libstdcxx_order(A + 1), libstdcxx_order(A)
        same = [p for p in full if p < A] == alone
        cfg = make_cfg(num_agents=A, mode_number=7, task_modes=task_bits([1, 7]), **MINI)
        if same:
            assert make_layout(cfg).P == A + 1
        else:
            with pytest.raises(AgarclError, match="player order of mode 1 differs"):
                make_layout(cfg)
        if A == 1:
            assert same


def test_ctypes_cfg_names_the_header_fields():
    from agarcl_b200._abi import Cfg, make_cfg
    assert C.sizeof(Cfg) == 28 * 4 and [f[0] for f in Cfg._fields_][-2:] == ["task_modes", "pixel_obs"]
    assert make_cfg(pixel_obs=32).pixel_obs == 32


def test_kernels_touched_by_tasks_have_no_spills():
    from agarcl_b200 import build
    flags = [f for f in build.NVCC_FLAGS if f != "-shared"]
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    text = ""
    with tempfile.TemporaryDirectory() as d:
        for src in ("reset_kernel.cu", "episode_kernel.cu"):
            r = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, src), "-o", os.path.join(d, "k.o")],
                               capture_output=True, text=True, check=True)
            text += r.stdout + r.stderr
    blocks = re.findall(r"Function properties for (\S*k_(?:reset|episode|set_tasks)\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill "
                        r"stores, (\d+) bytes spill loads", text)
    assert len(blocks) == 3, text
    for name, stack, st, ld in blocks:
        assert (int(stack), int(st), int(ld)) == (0, 0, 0), (name, stack, st, ld)
