"""Start states (agarcl_batch_set_start_states, the start mode of k_snapshot): every reset of an instance with a start slot
begins in the slot's game on the instance's own draw stream, and everything around the game (dones, episode counters, ram
records, observation, pictures, final observation) is what a reset does.  Checked against the oracle, against a twin batch
without a table, for every observation kind, for mixed-task batches, explicit resets, refusals and host waits."""
import ctypes as C

import numpy as np
import pytest

from agarcl_b200 import OBS_I16, RNG_MT19937, RNG_PHILOX, RNG_REPLAY, make_cfg
from agarcl_b200._abi import HDR_DT, StateView, task_bits
from gpu_parity_lib import SMALL, assert_no_host_wait, device_record, i32, philox_uniform_np

GRID_KW = [SMALL, dict(num_frames=2, grid_size=33, observe_others=False, obs_dtype=OBS_I16, ram_obs=1, **SMALL)]


def _actions(rng, n):
    return rng.uniform(-1, 1, size=(n, 2)).astype(np.float32), rng.integers(0, 3, size=n).astype(np.int32)


def _slot_blob(pool, slot, stride):
    return pool[slot, 64:64 + stride].cpu().numpy().copy()


def _patched(L, blob, seed, cursor):
    """the slot's blob as a start-state reset leaves it: the instance's seed and cursor, no respawn mask"""
    sv = StateView(L, blob.copy())
    h = sv.blob[L.off_hdr:L.off_hdr + 64].view(HDR_DT)
    h["seed_lo"], h["seed_hi"] = int(seed) & 0xFFFFFFFF, int(seed) >> 32
    h["rng_cursor"] = cursor
    h["respawned_lo"], h["respawned_hi"] = 0, 0
    return sv


def _aged(cfg, seeds, steps, rng):
    from agarcl_b200.batch import Batch
    b = Batch(cfg)
    b.seed(np.asarray(seeds, np.uint64))
    b.reset()
    for _ in range(steps):
        b.set_actions(*_actions(rng, b.N * b.A))
        b.step()
    return b


@pytest.mark.gpu
def test_start_states_against_the_oracle():
    """configs[1] under RNG_PHILOX with instance_base != 0, step_autoreset with 30-step episodes: one slot forked into three
    instances, one instance on its own slot, two spawning.  Every instance equals an oracle after every step; at each reset the
    oracle restarts from the slot's blob with the destination's seed and cursor (or spawns on its own stream).  Every instance
    plays the same action for the same step of its episode, so episodes and forks from one slot differ only where the game draws."""
    import torch
    from _helpers import Oracle, oracle_layout, oracle_lib, random_actions
    from agarcl_b200._abi import compare_states
    from agarcl_b200.batch import Batch
    oracle_lib().oracle_set_trig_mode(1)
    base, N, T, steps, limit, replay_len = 500, 6, 12, 200, 30, 1 << 17
    seeds = [101, 202, 303, 404, 505, 606]
    cfg = make_cfg(n_instances=N, rng_mode=RNG_PHILOX, instance_base=base)
    ocfg = make_cfg(n_instances=N, rng_mode=RNG_REPLAY, cap_replay=replay_len, instance_base=base)
    b = _aged(cfg, seeds, T, np.random.default_rng(3))
    A, L = b.A, b.layout
    pool = b.snapshot_pool(3)
    b.save_states(pool, i32([1, 3]), i32([0, 2]))
    slot_of = np.array([0, 0, 0, 2, -1, -1], np.int32)
    b.set_autoreset(limit, keep_final_obs=True)
    b.set_start_states(pool, i32(slot_of))
    ep, final_obs, res = b.episode(), b.final_obs(), b.start_result()
    torch.cuda.synchronize()
    slot_blobs = {s: _slot_blob(pool, s, L.stride) for s in (0, 2)}
    Lo = oracle_layout(ocfg)
    assert Lo.stride == L.stride
    oras = []
    for i in range(N):
        o = Oracle(ocfg, Lo)
        o.state.blob[:] = b.download_state(i).blob
        o.set_replay(philox_uniform_np(seeds[i], base + i, np.arange(replay_len)))
        oras.append(o)
    table = [random_actions(np.random.default_rng(100 + k), A) for k in range(limit + 1)]
    host_steps, acc = np.zeros(N, np.int64), np.zeros((N, A))
    starts = {i: [] for i in range(N)}  # (start cursor, blob 10 steps into the episode) of every start-state episode
    resets = 0
    for st in range(steps):
        acts = [table[host_steps[i]] for i in range(N)]
        b.set_actions(np.concatenate([a[0] for a in acts]), np.concatenate([a[1] for a in acts]))
        b.step_autoreset()
        torch.cuda.synchronize()
        g_rew, g_done = b.rewards_tensor().cpu().numpy().reshape(N, A), ep["done"].cpu().numpy().reshape(N, A)
        g_obs = b.obs_tensor().cpu().numpy().reshape(N, A, *b.obs_shape[1:])
        g_final = final_obs.cpu().numpy().reshape(N, A, *b.obs_shape[1:])
        mask, r = ep["reset_mask"].cpu().numpy().astype(bool), res.cpu().numpy()
        steps_dev, length, ret = ep["steps"].cpu().numpy(), ep["episode_length"].cpu().numpy(), ep["episode_return"].cpu().numpy()
        for i, o in enumerate(oras):
            o.set_actions(*acts[i])
            o_rew, o_done, o_obs = o.step(with_obs=True)
            done = o_done.astype(bool) | (host_steps[i] >= limit)
            host_steps[i] += 1
            acc[i] += o_rew
            assert np.array_equal(g_rew[i], o_rew) and np.array_equal(g_done[i], done.astype(np.uint8)), (st, i)
            assert mask[i] == done.any(), (st, i)
            if mask[i]:
                resets += 1
                assert np.array_equal(g_final[i], o_obs), f"step {st} inst {i}: final_obs"
                assert length[i] == host_steps[i] and np.array_equal(ret.reshape(N, A)[i], acc[i]), (st, i)
                host_steps[i], acc[i] = 0, 0.0
                if slot_of[i] >= 0:
                    cursor = int(o.state.hdr["rng_cursor"])
                    o.state.blob[:] = _patched(L, slot_blobs[slot_of[i]], seeds[i], cursor).blob
                    assert np.array_equal(b.download_state(i).blob, o.state.blob), f"step {st} inst {i}: start blob"
                    starts[i].append([cursor, None])
                else:
                    o.reset_keep_stream()
                o_obs = np.stack([o.obs(a) for a in range(A)])
            assert r[i] == (0 if not mask[i] or slot_of[i] < 0 else 1), (st, i, r[i])
            assert steps_dev[i] == host_steps[i], (st, i)
            gs = b.download_state(i)
            d = compare_states(o.state, gs)
            assert not d, f"step {st} inst {i}: {d[:6]}"
            assert int(gs.hdr["rng_cursor"]) == int(o.state.hdr["rng_cursor"]) and int(gs.hdr["flags"]) == int(o.state.hdr["flags"])
            assert np.array_equal(g_obs[i], o_obs), f"step {st} inst {i}: obs"
            if starts[i] and starts[i][-1][1] is None and host_steps[i] == 10:
                starts[i][-1][1] = gs.blob.copy()
    assert resets >= 3 * N, resets
    for i in (0, 1, 2, 3):
        assert len(starts[i]) >= 2, (i, starts[i])
        cursors = [c for c, _ in starts[i]]
        assert cursors == sorted(set(cursors)), f"inst {i}: a start reused its stream: {cursors}"
        assert not np.array_equal(starts[i][0][1], starts[i][1][1]), f"inst {i}: two episodes from one slot did not diverge"
    forks = [starts[i][0][1] for i in (0, 1, 2)]
    assert not np.array_equal(forks[0], forks[1]) and not np.array_equal(forks[1], forks[2]), "forks did not diverge"
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", GRID_KW)
def test_no_start_and_rejected_slots_are_a_spawn(kw):
    """three twins over many auto-resets: no table, a table of all -1, and a table whose every slot is rejected (unsaved slot
    with magic 0, out of range, another configuration's fingerprint): bit-identical, and start_result 2 exactly where the
    rejected batch reset"""
    import torch
    from agarcl_b200.batch import Batch
    N, limit = 12, 9
    cfg = make_cfg(n_instances=N, **kw)
    bs = [Batch(cfg) for _ in range(3)]
    for b in bs:
        b.seed(17)
        b.reset()
        b.set_autoreset(limit, keep_final_obs=True)
    pool = bs[2].snapshot_pool(3)  # slot 0 is never saved
    other = Batch(make_cfg(n_instances=2, **dict(kw, grid_size=64)))
    other.seed(1)
    other.reset()
    op = other.snapshot_pool(1)
    other.save_states(op, i32([1]))
    torch.cuda.synchronize()
    assert other.slot_bytes == bs[2].slot_bytes or kw is not SMALL
    w = min(other.slot_bytes, bs[2].slot_bytes)
    pool[1, :w] = op[0, :w]
    other.close()
    bs[1].set_start_states(bs[1].snapshot_pool(2), i32(np.full(N, -1)))
    bs[2].set_start_states(pool, i32(np.array([0, 1, 3, 99] * (N // 4))))
    rng = np.random.default_rng(21)
    resets = 0
    for t in range(40):
        acts = _actions(rng, N * bs[0].A)
        for b in bs:
            b.set_actions(*acts)
            b.step_autoreset()
        recs = [device_record(b) for b in bs]
        for k in recs[0]:
            assert np.array_equal(recs[0][k], recs[1][k]) and np.array_equal(recs[0][k], recs[2][k]), (t, k)
        m = recs[2]["reset_mask"].astype(bool)
        resets += int(m.sum())
        assert np.array_equal(bs[1].start_result().cpu().numpy(), np.zeros(N, np.uint8)), t
        assert np.array_equal(bs[2].start_result().cpu().numpy(), np.where(m, 2, 0)), t
    assert resets >= 3 * N
    for b in bs:
        b.close()


def _explicit_reset_case(kw, pixel=False):
    """a batch aged and saved, stepped on, then a table [slot 1, -1, slot 0, slot 3] and reset_device([1, 1, 1, 0])"""
    import torch
    N = 4
    cfg = make_cfg(n_instances=N, pixel_obs=64 if pixel else 0, **kw)
    seeds = [5, 6, 7, 8]
    b = _aged(cfg, seeds, 8, np.random.default_rng(8))
    b.set_autoreset(50, keep_final_obs=True)
    pool = b.snapshot_pool(4)
    b.save_states(pool, i32([0, 2, 3, 1]), i32([0, 1, 3, 2]))
    rng = np.random.default_rng(9)
    for _ in range(5):
        b.set_actions(*_actions(rng, N * b.A))
        b.step_autoreset()
    torch.cuda.synchronize()
    before = [b.download_state(i) for i in range(N)]
    rec = device_record(b)
    b.set_start_states(pool, i32([1, -1, 0, 3]))
    b.reset_device(i32([1, 1, 1, 0]).to(torch.uint8))
    torch.cuda.synchronize()
    want = {i: _patched(b.layout, _slot_blob(pool, s, b.layout.stride), seeds[i], int(before[i].hdr["rng_cursor"]))
            for i, s in ((0, 1), (2, 0))}
    return b, pool, rec, want


@pytest.mark.gpu
@pytest.mark.parametrize("kw", GRID_KW)
def test_explicit_resets_and_grid_observation(kw):
    """reset_device(mask) and reset() land in the table's slots: the blob is the patched slot, the grid observation the
    oracle's frame of it (earlier frames cleared), ram records cleared, episode counters restarted; outside the mask nothing
    changes"""
    import torch
    from _helpers import Oracle, oracle_layout, oracle_lib
    oracle_lib().oracle_set_trig_mode(1)
    b, pool, rec, want = _explicit_reset_case(kw)
    N, A, L = b.N, b.A, b.layout
    assert b.start_result().cpu().numpy().tolist() == [1, 0, 1, 0]
    after = device_record(b)
    ocfg = make_cfg(n_instances=N, rng_mode=RNG_REPLAY, cap_replay=1024, **kw)
    Lo = oracle_layout(ocfg)
    obs = after["obs"].reshape(N, A, *b.obs_shape[1:])
    C_ = L.obs_channels
    for i, sv in want.items():
        assert np.array_equal(after["blobs"][i], sv.blob), i
        o = Oracle(ocfg, Lo)
        o.state.blob[:] = sv.blob
        for a in range(A):
            frame = o.obs(a)
            if kw.get("obs_dtype") == OBS_I16:
                frame = np.clip(frame, -32768, 32767)
            assert np.array_equal(obs[i, a, -C_:], frame), (i, a)
            assert not obs[i, a, :-C_].any(), (i, a)
        if b.cfg.ram_obs:
            assert not after["ram"][i].any(), i
    for k in ("blobs", "ram", "steps"):
        if k in after:
            assert np.array_equal(after[k][3], rec[k][3]), k
    assert np.array_equal(obs[3], rec["obs"].reshape(N, A, *b.obs_shape[1:])[3])
    assert after["steps"].tolist()[:3] == [0, 0, 0] and after["steps"][3] == rec["steps"][3] > 0
    assert not after["dones"].reshape(N, A)[:3].any()
    # reset(): every instance, the host path; the result of the last restore is left alone
    restored = b.restore_states(pool, i32([0, -1, -1, 9]))
    b.set_start_states(pool, i32([2, 2, -1, 1]))
    b.reset()
    torch.cuda.synchronize()
    assert b.start_result().cpu().numpy().tolist() == [1, 1, 0, 1]
    assert restored.cpu().numpy().tolist() == [1, 0, 0, 2]
    assert np.array_equal(b.download_state(0).blob[L.off_players:], _slot_blob(pool, 2, L.stride)[L.off_players:])
    assert (b.episode()["steps"].cpu().numpy() == 0).all()
    b.close()


@pytest.mark.gpu
def test_pixels_after_a_start_state_reset():
    """with pixel_obs the picture of a started instance is oracle_draw's agent view of the patched blob; the final pictures of
    step_autoreset are those of the finished episode (a twin without a table)"""
    import torch
    from _helpers import AGENT, oracle_draw
    from agarcl_b200.batch import Batch
    b, pool, rec, want = _explicit_reset_case(SMALL, pixel=True)
    pics = b.pixels().cpu().numpy()
    for i, sv in want.items():
        for a in range(b.A):
            assert np.array_equal(pics[i * b.A + a], oracle_draw(b.cfg, b.layout, sv.blob, AGENT, a, 64)), (i, a)
    b.close()
    N, limit = 8, 6
    cfg = make_cfg(n_instances=N, pixel_obs=64, **dict(SMALL, num_bots=0))  # (no bot: every episode runs to the limit)
    x, y = Batch(cfg), Batch(cfg)
    for z in (x, y):
        z.seed(3)
        z.reset()
        z.set_autoreset(limit, keep_final_obs=True)
    pool = x.snapshot_pool(N)
    x.save_states(pool, i32(np.arange(N)))
    x.set_start_states(pool, i32(np.arange(N)[::-1].copy()))
    rng = np.random.default_rng(4)
    for t in range(limit + 1):
        acts = _actions(rng, N * x.A)
        for z in (x, y):
            z.set_actions(*acts)
            z.step_autoreset()
    torch.cuda.synchronize()
    m = x.episode()["reset_mask"].cpu().numpy().astype(bool)
    assert m.all() and (x.start_result().cpu().numpy() == 1).all()
    assert torch.equal(x.final_pixels(), y.final_pixels())
    for i in range(N):
        sv = x.download_state(i)
        for a in range(x.A):
            assert np.array_equal(x.pixels()[i * x.A + a].cpu().numpy(), oracle_draw(cfg, x.layout, sv.blob, AGENT, a, 64)), (i, a)
    x.close()
    y.close()


@pytest.mark.gpu
def test_mixed_task_start_states():
    """tasks [1, 7, 8]: a slot of mode 7 makes mode 7 current with the pending step limit, the pending mode stays; a slot whose
    mode is outside the set is rejected and the instance spawns its pending task"""
    import torch
    from agarcl_b200.batch import Batch
    N = 4
    cfg = make_cfg(n_instances=N, mode_number=1, task_modes=task_bits([1, 7, 8]), num_bots=0, arena_size=400, num_pellets=400)
    b = Batch(cfg)
    b.seed(2)
    b.set_tasks(i32([7, 1, 1, 1]))
    b.reset()
    b.set_autoreset(40)
    rng = np.random.default_rng(2)
    for _ in range(5):
        b.set_actions(*_actions(rng, N * b.A))
        b.step()
    pool = b.snapshot_pool(2)
    b.save_states(pool, i32([0, 0]), i32([0, 1]))
    torch.cuda.synchronize()
    pool[1, 28:32] = torch.tensor([10], dtype=torch.int32).view(torch.uint8).cuda()  # agarcl_snapshot_hdr.task_mode
    b.set_tasks(i32([-1, 8, 8, -1]), i32([0, 13, 14, 0]))
    b.set_start_states(pool, i32([-1, 0, 1, -1]))
    b.reset_device(i32([0, 1, 1, 0]).to(torch.uint8))
    torch.cuda.synchronize()
    tk = {k: v.cpu().numpy().tolist() for k, v in b.tasks().items()}
    assert b.start_result().cpu().numpy().tolist() == [0, 1, 2, 0]
    assert tk["mode"][1:3] == [7, 8] and tk["max_steps"][1:3] == [13, 14]
    assert tk["next_mode"][1:3] == [8, 8] and tk["next_max_steps"][1:3] == [13, 14]
    assert np.array_equal(b.download_state(1).blob[b.layout.off_players:],
                          _slot_blob(pool, 0, b.layout.stride)[b.layout.off_players:])
    sv = b.download_state(2)
    assert int(sv.hdr["tick"]) == 0 and int(sv.players["n_cells"][1]) == 1  # a fresh mode-8 game: its bot is spawned
    b.close()


@pytest.mark.gpu
def test_refusals_leave_the_table_and_nothing_waits():
    import torch
    from agarcl_b200._lib import AgarclError, lib
    from agarcl_b200.batch import Batch
    from agarcl_b200.env import BatchedGridEnvironment
    N = 4
    b = Batch(make_cfg(n_instances=N, **SMALL))
    pool = b.snapshot_pool(N)
    b.set_start_states(pool, i32([0, -1, 1, -1]))  # before the first reset: allowed
    b.seed(5)
    b.reset()
    assert b.start_result().cpu().numpy().tolist() == [2, 0, 2, 0]  # nothing saved yet
    b.save_states(pool, i32(np.arange(N)))
    sb = b.slot_bytes
    flat = torch.zeros(N * sb + 16, dtype=torch.uint8, device="cuda")
    misaligned = flat[1:1 + N * sb].view(N, sb)
    with pytest.raises(AgarclError, match="16-byte aligned"):
        b.set_start_states(misaligned, i32(np.arange(N)))
    with pytest.raises(AgarclError, match="int32"):
        b.set_start_states(pool, i32(np.arange(N)).long())
    with pytest.raises(AgarclError, match="4 entries"):
        b.set_start_states(pool, i32(np.arange(N + 1)))
    host = np.zeros(N * sb + 64, np.uint8)
    hp = (host.ctypes.data + 15) // 16 * 16
    idx = i32(np.arange(N))
    L, vp = lib(), C.c_void_p
    assert L.agarcl_batch_set_start_states(b._h, vp(hp), N, vp(idx.data_ptr()), None) != 0
    assert "device memory" in L.agarcl_last_error().decode()
    assert L.agarcl_batch_set_start_states(b._h, vp(pool.data_ptr()), 0, vp(idx.data_ptr()), None) != 0
    assert L.agarcl_batch_set_start_states(b._h, vp(pool.data_ptr()), N, None, None) != 0
    b.reset()
    torch.cuda.synchronize()
    assert b.start_result().cpu().numpy().tolist() == [1, 0, 1, 0]  # the table set before the refusals
    b.set_start_states(None)
    before = b.start_result().clone()
    b.reset()
    torch.cuda.synchronize()
    assert torch.equal(b.start_result(), before) and b._start_pool is None
    # launches of a plain step are those of a batch without a table
    c = Batch(make_cfg(n_instances=N, **SMALL))
    c.seed(5)
    c.reset()
    b.set_start_states(pool, i32(np.arange(N)))
    for z in (b, c):
        z.set_actions(*_actions(np.random.default_rng(1), N))
        z.step()
    assert b.launches_per_step() == c.launches_per_step()
    b.close()
    c.close()
    for kw, frag in ((dict(strict_reference=1, ticks_per_step=1), "strict_reference"), (dict(rng_mode=RNG_MT19937, cap_replay=4096), "MT19937")):
        x = Batch(make_cfg(n_instances=N, **kw, **SMALL))
        with pytest.raises(AgarclError, match=frag):
            x.set_start_states(x.snapshot_pool(N), idx)
        x.close()
    # no host wait: set_start_states and step_autoreset with a table
    M = 64
    env = BatchedGridEnvironment(M, num_bots=2, arena_size=200, num_pellets=100, num_viruses=2)
    env.seed(1)
    env.reset()
    env.set_autoreset(2, final_obs=True)
    epool = env.snapshot_pool(M)
    env.save_states(epool, i32(np.arange(M)))
    slots = i32(np.arange(M))
    s = torch.cuda.Stream()
    dxdy, act = torch.zeros((M, 2), device="cuda"), torch.zeros(M, dtype=torch.int32, device="cuda")
    for _ in range(4):
        env.set_start_states(epool, slots, stream=s.cuda_stream)
        env.step_autoreset(dxdy, act, stream=s.cuda_stream)

    def calls():
        env.set_start_states(epool, slots, stream=s.cuda_stream)
        for _ in range(3):
            env.step_autoreset(dxdy, act, stream=s.cuda_stream)

    assert_no_host_wait(calls, s)
    env.close()


@pytest.mark.gpu
def test_vector_env_start_states():
    """BatchedAgarioEnv: auto-resets and reset() begin in the chosen slots, info carries start_result, the new episode counts
    from 0 to the step limit"""
    import torch
    from agarcl_b200.gym_env import BatchedAgarioEnv
    N, limit = 8, 5
    env = BatchedAgarioEnv(N, num_bots=0, arena_size=200, num_pellets=100, num_viruses=2, number_steps=limit)
    env.seed(3)
    env.reset()
    zeros = lambda: (torch.zeros((N, 2), device="cuda"), torch.zeros(N, dtype=torch.int32, device="cuda"))  # noqa: E731
    for _ in range(3):
        env.step(*zeros())
    pool = env.snapshot_pool(N)
    env.save_states(pool, i32(np.arange(N)))
    env.set_start_states(pool, i32([0, 1, 2, 3, -1, -1, -1, -1]))
    for n in (limit - 3 + 1, limit + 1):  # the running episode ends, then the first one that began in the slots
        for k in range(n):
            _, _, _, _, info = env.step(*zeros())
            assert "start_result" in info and bool(info["reset_mask"].any()) == (k == n - 1), (n, k)
        assert bool(info["reset_mask"].all()) and info["start_result"].cpu().numpy().tolist() == [1] * 4 + [0] * 4
        assert (info["steps"].cpu().numpy() == 0).all() and (info["episode_length"].cpu().numpy() == limit + 1).all()
    env.reset()
    assert (env._env.batch.start_result().cpu().numpy() == [1] * 4 + [0] * 4).all()
    env.set_start_states(None)
    _, _, _, _, info = env.step(*zeros())
    assert "start_result" not in info
    env.close()
