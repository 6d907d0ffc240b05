"""Built-in bot policies for agents on the device (agarcl_batch_bot_actions, bot_kernel.cu): byte-exact against oracle_bot_decide
on downloaded blobs across configurations, ages and crafted states, the state left untouched, skipped and rejected agents, a
closed loop against the oracle, graph capture, the refusals, the Python layers and the task runner's bot policies."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from _helpers import ROOT, Oracle, oracle_bot_batch, oracle_bot_decide, oracle_layout, oracle_lib, random_actions
from agarcl_b200 import RNG_REPLAY, make_cfg
from agarcl_b200._abi import BOT_BAD_TYPE, BOT_DEAD, BOT_DECIDED, BOT_NO_PELLET, BOT_SKIPPED, compare_states
from gpu_parity_lib import SMALL, aged_batch, device_record, i32, step_random

CASES = ["c1", "c2", "c3", "c4_four_agents", "c5", "mode1", "mode7", "mode8", "mode9", "mode10", "mixed_tasks", "int16", "ram_obs2",
         "mt19937", "strict_reference"]


SENT_F, SENT_I, SENT_U8 = np.float32(-12345.5), -777, 0xEE


def _check(b, types):
    """device bot_actions of `types` [N*A] against oracle_bot_decide on the downloaded blobs, byte for byte, outputs prefilled
    with sentinels; the blobs are the same before and after the call.  Returns the statuses."""
    import torch
    NA = b.N * b.A
    types = np.asarray(types, np.int32)
    dxdy = torch.full((NA, 2), float(SENT_F), dtype=torch.float32, device="cuda")
    target = torch.full((NA, 2), float(SENT_F), dtype=torch.float32, device="cuda")
    act = torch.full((NA,), SENT_I, dtype=torch.int32, device="cuda")
    status = torch.full((NA,), SENT_U8, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    blobs = np.stack([b.download_state(i).blob for i in range(b.N)])
    out = b.bot_actions(i32(types), out=(dxdy, act, status), target=target)
    assert out[0] is dxdy and out[1] is act and out[2] is status
    torch.cuda.synchronize()
    after = np.stack([b.download_state(i).blob for i in range(b.N)])
    assert np.array_equal(blobs, after), "bot_actions changed the state"
    g = [t.cpu().numpy() for t in (dxdy, target, act, status)]
    o = oracle_bot_batch(b.cfg, b.layout, blobs, types)
    req = (types >= 0) & (types <= 3)
    assert np.array_equal(g[3], o[3]), f"status: {np.flatnonzero(g[3] != o[3])[:8]}"
    for k, what in ((0, "dxdy"), (1, "target")):
        gv, ov = g[k][req].view(np.uint32), o[k][req].view(np.uint32)
        if not np.array_equal(gv, ov):
            bad = np.flatnonzero(np.any(gv != ov, axis=1))
            j = np.flatnonzero(req)[bad[0]]
            raise AssertionError(f"{what} differs for {len(bad)} agents, first j={j} type {types[j]}: {g[k][j]} vs {o[k][j]}")
    assert np.array_equal(g[2][req], o[2][req]), "act"
    assert (g[0][~req] == SENT_F).all() and (g[1][~req] == SENT_F).all() and (g[2][~req] == SENT_I).all()
    return g[3]


def _all_types(b, rng):
    """every type for every agent, and one mix with skipped and invalid entries"""
    NA = b.N * b.A
    st = [_check(b, np.full(NA, t, np.int32)) for t in range(4)]
    mix = rng.choice([-1, 0, 1, 2, 3, 4, -2], NA).astype(np.int32)
    mix[0], mix[-1] = -1, 4
    st.append(_check(b, mix))
    return np.concatenate(st)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_bot_actions_match_oracle(name):
    """every agent and type at ages 0, 1 and 250"""
    b, rng, p_feed, p_split = aged_batch(name, second_reset=True)
    seen = set()
    for more in (0, 1, 249):
        step_random(b, rng, p_feed, p_split, more)
        seen |= set(_all_types(b, rng).tolist())
    assert BOT_DECIDED in seen and BOT_SKIPPED in seen and BOT_BAD_TYPE in seen
    if name == "c4_four_agents":  # the agents did split
        assert max(int(b.download_state(i).players["n_cells"][:b.A].max()) for i in range(b.N)) > 1
    b.close()


@pytest.mark.gpu
def test_aged_c2_multi_cell_and_popped_players():
    """c2 at 2000 steps: bots with many cells, players popped by viruses and eaten"""
    b, rng, pf, ps = aged_batch("c2", N=2, seed=11)
    step_random(b, rng, pf, ps, 2000)
    st = _all_types(b, rng)
    assert BOT_DECIDED in st
    L = b.layout
    sv = [b.download_state(i) for i in range(b.N)]
    assert max(int(s.players["n_cells"].max()) for s in sv) > 1
    assert sum(int(s.players["cells_eaten"].sum()) + int(s.players["viruses_eaten"].sum()) for s in sv) > 0
    assert L.P == 26
    b.close()


@pytest.mark.gpu
def test_crafted_states():
    """no pellets, tied pellet distances, a dead agent, and a 64-player instance with crowds to flee and chase"""
    from agarcl_b200.batch import Batch
    import torch
    b = Batch(make_cfg(n_instances=3, num_agents=4, num_bots=60, num_viruses=0, num_pellets=600, arena_size=300))
    b.seed(2)
    b.reset()
    L = b.layout
    assert L.P == 64
    rng = np.random.default_rng(4)
    # 0: crowded, players of every size within reach of each other, several cells each
    sv = b.download_state(0)
    for p in range(L.P):
        n = int(rng.integers(1, 6))
        sv.players["n_cells"][p] = n
        c = sv.cells[p][:n]
        c["x"], c["y"] = rng.uniform(120, 180, n), rng.uniform(120, 180, n)
        c["mass"] = rng.choice([20, 25, 30, 60, 100, 400, 2000], n)
    sv.players["action"][:] = rng.integers(0, 3, L.P)
    sv.players["n_cells"][2] = 0  # a dead agent
    b.upload_state(0, sv)
    # 1: no pellets
    sv = b.download_state(1)
    sv.hdr["n_pellets"] = 0
    b.upload_state(1, sv)
    # 2: pellets tied around every agent, one nearer than 0.01
    sv = b.download_state(2)
    k = 0
    for a in range(L.A):
        sv.cells[a][0]["x"], sv.cells[a][0]["y"] = 50.0 + 70.0 * a, 50.0 + 70.0 * a
        x, y = float(sv.cells[a][0]["x"]), float(sv.cells[a][0]["y"])
        for dx, dy in ((3, 4), (-4, 3), (4, -3), (0.004, 0), (-3, -4)):
            sv.pellets[k] = (x + dx, y + dy)
            k += 1
    # ... and the only player near agent 0 is far down the order (the second round of lanes): a bot with a cell agent 0 eats
    order = list(L.order[:L.P])
    near = [p for p in order[40:] if p >= L.A][0]
    for p in range(L.A, L.P):
        for i in range(int(sv.players["n_cells"][p])):
            sv.cells[p][i]["x"], sv.cells[p][i]["y"] = 290.0 - 0.1 * p, 290.0
    x0, y0 = float(sv.cells[0][0]["x"]), float(sv.cells[0][0]["y"])
    sv.cells[0][0]["mass"] = 100
    sv.players["n_cells"][near] = 1
    sv.cells[near][0]["x"], sv.cells[near][0]["y"], sv.cells[near][0]["mass"] = x0 + 8.0, y0 + 6.0, 40
    b.upload_state(2, sv)
    torch.cuda.synchronize()
    st = _all_types(b, rng).reshape(5, b.N, b.A)
    assert (st[:4, 1] == BOT_NO_PELLET).any() and (st[:4, 0, 2] == BOT_DEAD).all()
    assert (st[:4, 0][:, [0, 1, 3]] == BOT_DECIDED).all()
    tgt = torch.zeros((b.N * b.A, 2), device="cuda")
    b.bot_actions(1, target=tgt)  # HungryShy agent 0 of instance 2 flees from `near`
    assert tgt[2 * b.A].tolist() != [0.0, 0.0]
    d = oracle_bot_decide(b.cfg, L, b.download_state(2).blob, 0, 1)[1]
    assert np.allclose(d, [x0 - 8.0, y0 - 6.0], atol=1e-3) and np.array_equal(tgt[2 * b.A].cpu().numpy(), d)
    b.close()


@pytest.mark.gpu
def test_state_untouched_against_a_twin():
    """the batch that computes bot actions every step stays identical to a twin that never does, over 50 steps"""
    from agarcl_b200.batch import Batch
    cfg = make_cfg(n_instances=6, num_agents=2, **SMALL)
    twins = [Batch(cfg), Batch(cfg)]
    for b in twins:
        b.seed(8)
        b.reset()
    rng = np.random.default_rng(0)
    types = i32(rng.choice([-1, 0, 1, 2, 3, 9], cfg.n_instances * 2))
    for t in range(50):
        dxdy, act = random_actions(rng, cfg.n_instances * 2)
        before = device_record(twins[0])
        for ty in (types, 0, 1, 2, 3):
            twins[0].bot_actions(ty)
        after = device_record(twins[0])
        for k in before:
            assert np.array_equal(before[k], after[k]), f"step {t}: bot_actions changed {k}"
        for b in twins:
            b.set_actions(dxdy, act)
            b.step()
        a, c = device_record(twins[0]), device_record(twins[1])
        for k in a:
            assert np.array_equal(a[k], c[k]), f"step {t}: {k} differs from the twin"


@pytest.mark.gpu
def test_closed_loop_against_the_oracle():
    """300 steps with the device's bot actions fed to set_actions(on_device) and the oracle driven by oracle_bot_decide: states,
    rewards, dones and observations identical after every step.  Instance 1 has an agent driven by a random policy (type -1:
    its entries of the action buffer are the policy's)"""
    import torch
    from agarcl_b200.batch import Batch
    oracle_lib().oracle_set_trig_mode(1)
    seeds = [21, 22]
    n, A = len(seeds), 4
    cfg = make_cfg(n_instances=n, rng_mode=RNG_REPLAY, cap_replay=1 << 16, num_agents=A, **SMALL)
    b = Batch(cfg)
    L = b.layout
    Lo = oracle_layout(cfg)
    assert bytes(L) == bytes(Lo)
    oras = []
    for i, s in enumerate(seeds):
        o = Oracle(cfg, Lo)
        o.seed_mt(s, 1 << 16)
        b.set_replay(i, o.replay)
        oras.append(o)
    b.seed(np.asarray(seeds, np.uint64))
    b.reset()
    for o in oras:
        o.reset()
    types = np.array([0, 1, 2, 3, 3, -1, 1, 2], np.int32)
    types_t = i32(types)
    dxdy_t = torch.zeros((n * A, 2), dtype=torch.float32, device="cuda")
    act_t = torch.zeros(n * A, dtype=torch.int32, device="cuda")
    status_t = torch.zeros(n * A, dtype=torch.uint8, device="cuda")
    b.set_actions_device(dxdy_t.data_ptr(), act_t.data_ptr())
    obs_t, rew_t, done_t = b.obs_tensor(), b.rewards_tensor(), b.dones_tensor()
    rng = np.random.default_rng(3)
    seen = set()
    for st in range(300):
        rdxdy, ract = random_actions(rng, n * A)
        dxdy_t.copy_(torch.from_numpy(rdxdy))
        act_t.copy_(torch.from_numpy(ract))
        b.bot_actions(types_t, out=(dxdy_t, act_t, status_t))
        b.step()
        torch.cuda.synchronize()
        g_dxdy, g_act, g_obs = dxdy_t.cpu().numpy(), act_t.cpu().numpy(), obs_t.cpu().numpy().reshape(n, A, *b.obs_shape[1:])
        g_rew, g_done = rew_t.cpu().numpy().reshape(n, A), done_t.cpu().numpy().reshape(n, A)
        seen |= set(status_t.cpu().numpy().tolist())
        for i, o in enumerate(oras):
            o_dxdy, o_act = rdxdy[i * A:(i + 1) * A].copy(), ract[i * A:(i + 1) * A].copy()
            for a in range(A):
                if types[i * A + a] >= 0:
                    d, _, ac, _ = oracle_bot_decide(cfg, Lo, o.state.blob, a, types[i * A + a])
                    o_dxdy[a], o_act[a] = d, ac
            assert np.array_equal(o_dxdy.view(np.uint32), g_dxdy[i * A:(i + 1) * A].view(np.uint32)), f"step {st} inst {i}: dxdy"
            assert np.array_equal(o_act, g_act[i * A:(i + 1) * A]), f"step {st} inst {i}: act"
            o.set_actions(o_dxdy, o_act)
            o_rew, o_done, o_obs = o.step(with_obs=True)
            gs = b.download_state(i)
            d = compare_states(o.state, gs)
            assert not d, f"step {st} inst {i}: {d[:6]}"
            assert int(gs.hdr["flags"]) == int(o.state.hdr["flags"]), (st, i)
            assert np.array_equal(g_rew[i], o_rew) and np.array_equal(g_done[i], o_done), f"step {st} inst {i}: rewards / dones"
            assert np.array_equal(g_obs[i], o_obs), f"step {st} inst {i}: observation"
    assert BOT_DECIDED in seen and BOT_SKIPPED in seen
    b.close()


@pytest.mark.gpu
def test_graph_capture_of_bot_actions_and_step_autoreset():
    """bot_actions -> step_autoreset captured in a CUDA graph (capture fails on any synchronising call); replaying it equals the
    eager run of a twin batch, step for step"""
    import torch
    from agarcl_b200.batch import Batch
    cfg = make_cfg(n_instances=8, num_agents=2, **SMALL)
    twins = [Batch(cfg), Batch(cfg)]
    types = i32(np.random.default_rng(1).choice([-1, 0, 1, 2, 3], 16))
    bufs = []
    for b in twins:
        b.seed(3)
        b.reset()
        b.set_autoreset(40)
        buf = (torch.zeros((16, 2), dtype=torch.float32, device="cuda"), torch.zeros(16, dtype=torch.int32, device="cuda"),
               torch.zeros(16, dtype=torch.uint8, device="cuda"))
        b.set_actions_device(buf[0].data_ptr(), buf[1].data_ptr())
        bufs.append(buf)
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for b, buf in zip(twins, bufs):  # warm-up, one step each
            b.bot_actions(types, out=buf)
            b.step_autoreset(stream=s.cuda_stream)
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        twins[1].bot_actions(types, out=bufs[1])
        twins[1].step_autoreset(stream=s.cuda_stream)
    torch.cuda.synchronize()
    for t in range(60):
        twins[0].bot_actions(types, out=bufs[0])
        twins[0].step_autoreset()
        g.replay()
        a, c = device_record(twins[0]), device_record(twins[1])
        for k in a:
            assert np.array_equal(a[k], c[k]), f"replay {t}: {k}"
        for x, y in zip(bufs[0], bufs[1]):
            assert torch.equal(x, y), f"replay {t}: outputs"


@pytest.mark.gpu
def test_refusals_enqueue_nothing():
    import torch
    from agarcl_b200 import _lib
    from agarcl_b200.batch import Batch
    L = _lib.lib()
    vp = C.c_void_p
    cfg = make_cfg(n_instances=2, num_agents=2, **SMALL)
    fresh = Batch(cfg)
    types = i32([0, 1, 2, 3])
    dxdy = torch.full((5, 2), 7.0, dtype=torch.float32, device="cuda")
    target = torch.full((5, 2), 7.0, dtype=torch.float32, device="cuda")
    act = torch.full((4,), 7, dtype=torch.int32, device="cuda")
    status = torch.full((4,), 7, dtype=torch.uint8, device="cuda")

    def untouched():
        torch.cuda.synchronize()
        return bool((dxdy == 7).all() and (target == 7).all() and (act == 7).all() and (status == 7).all())

    def refused(b, t, d, a, tg, s, text, rc=-1):
        got = L.agarcl_batch_bot_actions(b._h, vp(t), vp(d), vp(a), vp(tg), vp(s), None)
        assert got == rc, (got, text)
        assert text in L.agarcl_last_error().decode(), L.agarcl_last_error().decode()
        assert untouched(), f"{text}: output written"

    ok = (types.data_ptr(), dxdy.data_ptr(), act.data_ptr(), target.data_ptr(), status.data_ptr())
    refused(fresh, *ok, "before reset", rc=-4)
    b = Batch(cfg)
    b.seed(1)
    b.reset()
    for k in range(3):
        args = list(ok)
        args[k] = 0
        refused(b, *args, "null")
    for k in (1, 3):
        args = list(ok)
        args[k] += 4
        refused(b, *args, "8-byte aligned")
    host = np.zeros(64, np.float32)
    hp = (host.ctypes.data + 15) & ~15
    pinned = torch.zeros(64, dtype=torch.float32).pin_memory()
    for k, what in enumerate(("type", "dxdy", "act", "target", "status")):
        for p in (hp, pinned.data_ptr()):
            args = list(ok)
            args[k] = p
            refused(b, *args, f"the {what} array")
    assert not host.any() and not pinned.any()
    with pytest.raises(_lib.AgarclError, match="int32"):
        b.bot_actions(torch.zeros(4, dtype=torch.int64, device="cuda"))
    with pytest.raises(_lib.AgarclError, match="4 entries"):
        b.bot_actions(i32([0, 1, 2]))
    with pytest.raises(_lib.AgarclError, match="act"):
        b.bot_actions(0, out=(dxdy[:4], act[:3], status))
    assert untouched()
    # the optional outputs may be NULL
    assert L.agarcl_batch_bot_actions(b._h, vp(types.data_ptr()), vp(dxdy.data_ptr()), vp(act.data_ptr()), None, None, None) == 0
    torch.cuda.synchronize()
    assert not (dxdy[:4] == 7).all() and (dxdy[4] == 7).all() and (target == 7).all() and (status == 7).all()


@pytest.mark.gpu
def test_python_layers():
    """Batch (int and tensor types, out=), BatchedGridEnvironment and BatchedAgarioEnv; the outputs go straight into step()"""
    import torch
    from agarcl_b200 import BOT_AGGRESSIVE, BOT_HUNGRY, BOT_TYPES, BatchedGridEnvironment
    from agarcl_b200.gym_env import BatchedAgarioEnv
    env = BatchedAgarioEnv(4, num_agents=2, num_bots=4, arena_size=300, num_pellets=300, num_viruses=4)
    env.seed(3)
    env.reset()
    b = env._env.batch
    for _ in range(5):
        dxdy, act, status = env.bot_actions(BOT_HUNGRY)
        assert dxdy.shape == (8, 2) and dxdy.dtype == torch.float32 and act.dtype == torch.int32 and status.dtype == torch.uint8
        obs, rew, done, trunc, info = env.step(dxdy, act)
    ref = b.bot_actions(i32([BOT_HUNGRY] * 8))
    got = env.bot_actions(BOT_HUNGRY)
    for x, y in zip(ref, got):
        assert torch.equal(x, y)
    buf = (torch.zeros((8, 2), device="cuda"), torch.zeros(8, dtype=torch.int32, device="cuda"),
           torch.zeros(8, dtype=torch.uint8, device="cuda"))
    out = env.bot_actions(i32([BOT_AGGRESSIVE, -1] * 4), out=buf)
    assert all(x is y for x, y in zip(out, buf))
    assert (buf[2][1::2] == BOT_SKIPPED).all() and (buf[0][1::2] == 0).all() and (buf[2][0::2] != BOT_SKIPPED).all()
    torch.cuda.synchronize()
    _check(b, [BOT_TYPES["aggressive_shy"]] * 8)
    env.close()

    g = BatchedGridEnvironment(3, num_agents=1, num_bots=2, arena_size=200, num_pellets=100, num_viruses=0)
    g.seed(5)
    g.reset()
    tgt = torch.zeros((3, 2), device="cuda")
    dxdy, act, status = g.bot_actions(BOT_TYPES["hungry"], target=tgt)
    obs, rew, done = g.step(dxdy, act)
    torch.cuda.synchronize()
    assert (status == BOT_DECIDED).all() and torch.isfinite(tgt).all()
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mixed", [False, True])
def test_run_tasks_configs_with_a_bot_policy(mixed):
    cmd = [sys.executable, os.path.join(ROOT, "tools", "run_tasks_configs.py"), "--policy", "hungry", "--steps", "50", "--envs", "64"]
    if mixed:
        cmd.append("--mixed")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [json.loads(x) for x in r.stdout.splitlines() if x.startswith("{")]
    assert len(lines) == (11 if mixed else 10)
    assert all(x["policy"] == "hungry" for x in lines)
