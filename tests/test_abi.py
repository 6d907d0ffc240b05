"""CPU: the C-ABI library loads, exports every symbol include/agarcl_b200.h declares and the ctypes binding binds exactly
those, derives the same layout as the oracle's independent restatement, and reports errors the way the reference does."""
import ctypes as C
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from _helpers import ROOT, oracle_layout, oracle_lib
from agarcl_b200 import _lib, make_cfg
from agarcl_b200._abi import Archive, ArchiveCfg, Cfg, Layout


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "agarcl_b200.h")).read()
    return sorted(set(re.findall(r"\b(agarcl_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    lib = _lib.lib()
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/agarcl_b200.h but not exported"
        assert getattr(lib, s).argtypes is not None, f"{s} is not bound"
    assert set(_lib.SYMBOLS) == set(syms)
    assert b"sm_100a" in lib.agarcl_version()


def test_struct_sizes_match_header():
    assert C.sizeof(Cfg) == 28 * 4
    assert C.sizeof(Layout) == (7 + 7 + 5 + 64 + 64) * 4
    assert C.sizeof(ArchiveCfg) == 24
    assert C.sizeof(Archive) == 10 * 8 + 16


@pytest.mark.parametrize("kw", [dict(), dict(num_agents=4, num_bots=8), dict(num_bots=40, num_agents=3),
                                dict(mode_number=1, arena_size=350, num_pellets=500, num_bots=0),
                                dict(mode_number=8, num_bots=1), dict(mode_number=5, arena_size=350, num_pellets=100),
                                dict(num_bots=0, num_viruses=0, observe_pellets=False), dict(rng_mode=1, cap_replay=777)])
def test_layout_matches_oracle_restatement(kw):
    cfg = make_cfg(**kw)
    a, b = _lib.make_layout(cfg), oracle_layout(cfg)
    assert bytes(a) == bytes(b)
    assert a.stride % 128 == 0 and a.off_pellets % 16 == 0


def test_player_order_is_libstdcxx_unordered_map_order():
    # SURVEY Appendix C: N <= 13 -> descending; N = 14 -> 13 0 1 ... 12; N = 26 -> 25..13 0..12
    L = _lib.make_layout(make_cfg(num_bots=12))
    assert list(L.order)[:13] == list(range(12, -1, -1))
    L = _lib.make_layout(make_cfg(num_bots=13))
    assert list(L.order)[:14] == [13] + list(range(13))
    L = _lib.make_layout(make_cfg(num_bots=25))
    assert list(L.order)[:26] == list(range(25, 12, -1)) + list(range(13))
    L = _lib.make_layout(make_cfg(num_bots=29))
    assert list(L.order)[:30] == [29] + list(range(12, -1, -1)) + list(range(13, 29))


def test_bot_roster_quirk_q14():
    L = _lib.make_layout(make_cfg(num_agents=2, num_bots=7))
    assert list(L.bot_type)[:9] == [-1, -1, 0, 1, 2, 3, 0, 0, 0]
    L = _lib.make_layout(make_cfg(mode_number=9, num_bots=5))  # modes 7..10: exactly one bot of type mode-7
    assert L.P == 2 and list(L.bot_type)[:2] == [-1, 2]
    L = _lib.make_layout(make_cfg(mode_number=4, num_bots=5))  # no bots outside mode 0 / 7..10
    assert L.P == 1


def test_invalid_configs_are_rejected_with_a_message():
    for kw, frag in [(dict(mode_number=11), "mode"), (dict(ticks_per_step=0), "ticks_per_step"),
                     (dict(num_agents=0), "num_agents"), (dict(num_bots=64), "too many players")]:
        with pytest.raises(_lib.AgarclError) as e:
            _lib.make_layout(make_cfg(**kw))
        assert frag in str(e.value)


def test_mt19937_stream_product_vs_oracle():
    n = 4096
    for seed in (0, 1, 42, 2**31 + 5):
        a = np.zeros(n, np.float32)
        b = np.zeros(n, np.float32)
        _lib.check(_lib.lib().agarcl_mt19937_draws(C.c_uint64(seed), a.ctypes.data_as(C.c_void_p), n))
        oracle_lib().oracle_mt19937_draws(C.c_uint64(seed), b.ctypes.data_as(C.c_void_p), n)
        assert np.array_equal(a, b)
        assert (a >= 0).all() and (a < 1).all()


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from agarcl_b200.batch import Batch
    with pytest.raises(_lib.AgarclError) as e:
        Batch(make_cfg())
    assert "no CPU path" in str(e.value)


def test_take_actions_size_check_like_reference():
    # BaseEnvironment::take_actions throws when len(actions) != num_agents (BaseEnvironment.hpp:142-144)
    from agarcl_b200.env import GridEnvironment
    env = GridEnvironment(2, 4, 1000, True, 1000, 25, 25, 1, 0, 0)
    with pytest.raises(RuntimeError) as e:
        env.take_actions([(0.0, 0.0, 0)])
    assert "does not match number of agents" in str(e.value)
    assert env.observation_shape() == (8, 128, 128)
    env.configure_observation({"grid_size": 64, "observe_others": False, "num_frames": 2})
    assert env.observation_shape() == (12, 64, 64)


def test_host_buffer_checks_hold_under_python_O():
    """Batch refuses host arrays of the wrong size before the library reads them: the checks are no asserts, so `python -O`
    keeps them.  (Batch.__new__: no library batch is needed, each call is refused before it would reach one.)"""
    script = textwrap.dedent("""
        import numpy as np
        from agarcl_b200._abi import Layout, StateView
        from agarcl_b200._lib import AgarclError
        from agarcl_b200.batch import Batch
        b = Batch.__new__(Batch)
        b.N, b.A = 3, 2
        b.layout = Layout(stride=256)
        calls = {"short dxdy": lambda: b.set_actions(np.zeros((5, 2), np.float32), np.zeros(6, np.int32)),
                 "short act": lambda: b.set_actions(np.zeros((6, 2), np.float32), np.zeros(5, np.int32)),
                 "short reset mask": lambda: b.reset(np.ones(2, np.uint8)),
                 "short state": lambda: b.upload_state(0, StateView(Layout(stride=128)))}
        for what, call in calls.items():
            try:
                call()
            except AgarclError:
                continue
            raise SystemExit(what + " was not refused")
    """)
    r = subprocess.run([sys.executable, "-O", "-c", script], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_compiled_agarcl_module_surface():
    """The pybind11 module `agarcl` (agarcl_b200/csrc/pybind_agarcl.cpp) is compiled, imports by the reference's name, and
    exposes the classes / methods environment/bindings.cpp:94-135,181-374 binds; errors come back as RuntimeError."""
    import agarcl
    assert agarcl.has_screen_env is False
    for cls in ("GridEnvironment", "GoBiggerEnvironment", "FoodInfo", "VirusInfo", "SporeInfo", "CloneInfo", "GlobalState",
                "PlayerState", "PlayerStates"):
        assert hasattr(agarcl, cls), cls
    for m in ("seed", "configure_observation", "observation_shape", "dones", "take_actions", "reset", "render", "step", "get_state",
              "get_frame", "close", "save_env_state"):
        assert hasattr(agarcl.GridEnvironment, m), m
    for m in ("configure_observation", "get_state", "take_actions", "dones", "observation_shape", "seed", "reset", "step", "render",
              "close", "load_env_state", "save_env_state"):
        assert hasattr(agarcl.GoBiggerEnvironment, m), m
    env = agarcl.GridEnvironment(2, 4, 1000, True, 1000, 25, 25, 1, 0, 0)
    assert env.observation_shape() == (8, 128, 128)
    env.configure_observation({"grid_size": 64, "observe_others": False, "num_frames": 2})
    assert env.observation_shape() == (12, 64, 64)
    with pytest.raises(RuntimeError):
        agarcl.GridEnvironment(1, 4, 1000, True, 1000, 25, 25, 1, 0, 11)  # Engine::set_mode throws on a bad mode
    with pytest.raises(TypeError):
        agarcl.GridEnvironment(1, 4)  # the ten positional arguments of bindings.cpp:102
    g = agarcl.GoBiggerEnvironment(512, 512, 1000, 1, 4, 300, True, 200, 4, 5, 1)  # defaults: c_death, mode_number, load_env_snapshot, agent_view
    assert g.observation_shape() == (0, 512, 512)
    gs = agarcl.GlobalState(width=3, height=4, frame_limit=5, last_frame=0, team_num=2)
    assert str(gs) == "GlobalState(map_width=3, map_height=4, frame_limit=5, team_num=2)"
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU path"):
            env.reset()
