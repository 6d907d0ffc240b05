"""Snapshot pools (agarcl_batch_save_states / agarcl_batch_restore_states, snapshot_kernel.cu): a restored instance steps
bit for bit as the saved one did, a fork follows the oracle on the destination's draw stream, every other instance is left
untouched, bad slots are rejected per instance on the device, bad calls are refused before anything is enqueued, and
nothing makes the host wait."""
import ctypes as C
import io

import numpy as np
import pytest

from agarcl_b200 import OBS_I16, RNG_MT19937, RNG_PHILOX, RNG_REPLAY, make_cfg
from gpu_parity_lib import CASES, SMALL, assert_no_host_wait, device_record, i32

RT_CASES = ["mode9_deaths_and_limit", "configs1_two_agents", "int16", "two_frames", "ram_obs1", "ram_obs2"]


def _blobs(b):
    return np.stack([b.download_state(i).blob for i in range(b.N)])


def _record(b):
    """device_record with the episode results of the instances the last step reset only (the others hold an earlier
    episode's, which a restore does not bring back)"""
    r = device_record(b)
    mask = r["reset_mask"].astype(bool)
    r["episode_return"] = r["episode_return"].reshape(b.N, b.A)[mask]
    r["episode_length"] = r["episode_length"][mask]
    if "final_obs" in r:
        r["final_obs"] = r["final_obs"].reshape(b.N, -1)[mask]
    if "final_ram" in r:
        r["final_ram"] = r["final_ram"][mask]
    return r


def _assert_equal(a, b, what, keys=None, rows=None):
    for k in keys or a:
        x, y = a[k], b[k]
        if rows is not None and k in ("blobs", "ram", "steps"):
            x, y = x[rows], y[rows]
        elif rows is not None and k in ("obs", "rewards", "dones"):
            A = x.shape[0] // rows.size
            x, y = x.reshape(rows.size, A, -1)[rows], y.reshape(rows.size, A, -1)[rows]
        assert np.array_equal(x, y), f"{what}: {k} differs"


def _actions(rng, n):
    return rng.uniform(-1, 1, size=(n, 2)).astype(np.float32), rng.integers(0, 3, size=n).astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("name", RT_CASES)
def test_round_trip(name):
    """step T, save all, step K recording everything, restore all, step the same K actions: bit-identical at every step"""
    from agarcl_b200.batch import Batch
    N, T, K = 16, 20, 40
    cfg = make_cfg(n_instances=N, **CASES[name][0])
    b = Batch(cfg)
    b.seed(99)
    b.reset()
    b.set_autoreset(37, keep_final_obs=True)
    rng = np.random.default_rng(5)
    acts = [_actions(rng, N * b.A) for _ in range(T + K)]
    for t in range(T):
        b.set_actions(*acts[t])
        b.step_autoreset()
    pool = b.snapshot_pool(N)
    idx = i32(np.arange(N))
    b.save_states(pool, idx)
    at_save = _record(b)
    first, resets = [], 0
    for t in range(T, T + K):
        b.set_actions(*acts[t])
        b.step_autoreset()
        first.append(_record(b))
        resets += int(first[-1]["reset_mask"].sum())
    assert resets > 0, "no episode ended inside the window"
    res = b.restore_states(pool, idx)
    after = _record(b)
    assert after is not None and (res.cpu().numpy() == 1).all()
    _assert_equal(at_save, after, "after restore", keys=[k for k in ("blobs", "obs", "ram", "steps") if k in after])
    assert not after["rewards"].any() and not after["dones"].any()  # zeroed, like after a reset
    for t in range(T, T + K):
        b.set_actions(*acts[t])
        b.step_autoreset()
        _assert_equal(first[t - T], _record(b), f"{name} step {t}")
    b.close()


@pytest.mark.gpu
def test_fork_against_oracle():
    """configs[1] under RNG_PHILOX with instance_base != 0: instance j saved at step T and restored into the other instances
    steps like an oracle started from j's blob and fed the DESTINATION's Philox stream (seed_j, instance_base + i, cursor)"""
    import torch
    from _helpers import Oracle, oracle_layout, oracle_lib, random_actions
    from agarcl_b200._abi import compare_states
    from agarcl_b200.batch import Batch
    from gpu_parity_lib import philox_uniform_np
    oracle_lib().oracle_set_trig_mode(1)
    base, N, j, T, K, replay_len = 1000, 4, 1, 15, 50, 1 << 16
    cfg = make_cfg(n_instances=N, rng_mode=RNG_PHILOX, instance_base=base)
    ocfg = make_cfg(n_instances=N, rng_mode=RNG_REPLAY, cap_replay=replay_len, instance_base=base)
    b = Batch(cfg)
    seeds = [11, 22, 33, 44]
    b.seed(np.asarray(seeds, np.uint64))
    b.reset()
    A = b.A
    rng = np.random.default_rng(1)
    for _ in range(T):
        b.set_actions(*_actions(rng, N * A))
        b.step()
    pool = b.snapshot_pool(2)
    b.save_states(pool, i32([j]), i32([1]))
    torch.cuda.synchronize()
    src_blob = b.download_state(j).blob.copy()
    src_obs = b.obs_tensor()[j * A:(j + 1) * A].clone()
    res = b.restore_states(pool, i32([1, -1, 1, 1]))
    torch.cuda.synchronize()
    assert res.tolist() == [1, 0, 1, 1]
    obs = b.obs_tensor()
    for i in range(N):  # the re-rendered frame is the one the step showed
        assert torch.equal(obs[i * A:(i + 1) * A], src_obs), i
        assert np.array_equal(b.download_state(i).blob, src_blob), i
    Lo = oracle_layout(ocfg)
    assert Lo.stride == b.layout.stride
    oras = []
    for i in range(N):
        o = Oracle(ocfg, Lo)
        o.state.blob[:] = src_blob
        o.set_replay(philox_uniform_np(seeds[j], base + i, np.arange(replay_len)))
        oras.append(o)
    arng = np.random.default_rng(2)
    for st in range(K):
        dxdy, act = random_actions(arng, A)  # identical actions for every child
        b.set_actions(np.tile(dxdy, (N, 1)), np.tile(act, N))
        b.step()
        torch.cuda.synchronize()
        g_rew = b.rewards_tensor().cpu().numpy().reshape(N, A)
        g_done = b.dones_tensor().cpu().numpy().reshape(N, A)
        g_obs = b.obs_tensor().cpu().numpy().reshape(N, A, *b.obs_shape[1:])
        for i, o in enumerate(oras):
            o.set_actions(dxdy, act)
            o_rew, o_done, o_obs = o.step(with_obs=True)
            gs = b.download_state(i)
            d = compare_states(o.state, gs)
            assert not d, f"step {st} inst {i}: {d[:6]}"
            assert int(gs.hdr["rng_cursor"]) == int(o.state.hdr["rng_cursor"]) and int(gs.hdr["flags"]) == int(o.state.hdr["flags"])
            assert np.array_equal(g_rew[i], o_rew) and np.array_equal(g_done[i], o_done), (st, i)
            assert np.array_equal(g_obs[i], o_obs), f"step {st} inst {i}: obs"
    blobs = _blobs(b)
    assert any(not np.array_equal(blobs[0], blobs[i]) for i in range(1, N)), "the children did not diverge where the game draws"
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [SMALL, dict(num_frames=2, grid_size=33, observe_others=False, obs_dtype=OBS_I16, ram_obs=1, **SMALL)])
def test_partial_restore_leaves_the_others_untouched(kw):
    """a batch that restores some instances (one slot forked into two of them) and a twin that never restores: every other
    instance stays bit-identical, at the restore and over the following steps"""
    from agarcl_b200.batch import Batch
    N = 24
    cfg = make_cfg(n_instances=N, **kw)
    a, b = Batch(cfg), Batch(cfg)
    for x in (a, b):
        x.seed(7)
        x.reset()
        x.set_autoreset(30, keep_final_obs=True)
    rng = np.random.default_rng(9)
    pool = a.snapshot_pool(N)
    for t in range(30):
        acts = _actions(rng, N * a.A)
        for x in (a, b):
            x.set_actions(*acts)
            x.step_autoreset()
        if t == 10:
            a.save_states(pool, i32(np.arange(N)))
    slot_of = np.full(N, -1, np.int32)
    slot_of[[0, 5, 6, 17]] = [3, 5, 5, 20]
    res = a.restore_states(pool, i32(slot_of)).cpu().numpy()
    assert np.array_equal(res, np.where(slot_of >= 0, 1, 0))
    keep = slot_of < 0
    ra, rb = _record(a), _record(b)
    _assert_equal(ra, rb, "at the restore", keys=[k for k in ("blobs", "obs", "ram", "rewards", "dones", "steps") if k in ra], rows=keep)
    # the restored instances hold the slots' blobs (slot layout: the blob at byte 64)
    S = a.layout.stride
    p = pool.cpu().numpy()
    for i in np.flatnonzero(~keep):
        assert np.array_equal(ra["blobs"][i], p[slot_of[i], 64:64 + S]), i
    assert np.array_equal(ra["blobs"][5], ra["blobs"][6])
    for t in range(10):
        acts = _actions(rng, N * a.A)
        for x in (a, b):
            x.set_actions(*acts)
            x.step_autoreset()
        ra, rb = _record(a), _record(b)
        _assert_equal(ra, rb, f"step {t} after the restore", keys=[k for k in ("blobs", "obs", "ram", "rewards", "dones", "steps") if k in ra],
                      rows=keep)
    a.close()
    b.close()


@pytest.mark.gpu
def test_rejections_and_acceptance():
    import torch
    from agarcl_b200.batch import Batch
    N = 8
    cfg = make_cfg(n_instances=N, ram_obs=1, **SMALL)
    b = Batch(cfg)
    b.seed(3)
    b.reset()
    rng = np.random.default_rng(4)
    for _ in range(5):
        b.set_actions(*_actions(rng, N))
        b.step()
    sb = b.slot_bytes
    pool = b.snapshot_pool(6)  # slot 0 stays zero
    grid_kw = dict(grid_size=64, ram_obs=1, **SMALL)
    for k, other_kw in ((1, dict(mode_number=1, num_bots=0, arena_size=300, num_pellets=300, num_viruses=4, ram_obs=1)), (2, grid_kw)):
        o = Batch(make_cfg(n_instances=2, **other_kw))
        o.seed(1)
        o.reset()
        op = o.snapshot_pool(1)
        o.save_states(op, i32([1]))
        torch.cuda.synchronize()
        w = min(sb, o.slot_bytes)
        pool[k, :w] = op[0, :w]
        if k == 2:
            assert o.slot_bytes == sb  # only the fingerprint tells them apart
        o.close()
    assert grid_kw["grid_size"] != cfg.grid_size
    b.save_states(pool, i32([0, N + 3]), i32([3, 4]))  # slot 4: a source out of range
    snapshot = pool.clone()
    b.save_states(pool, i32([2]), i32([99]))  # a slot out of range is skipped
    torch.cuda.synchronize()
    assert torch.equal(pool, snapshot)
    assert int(pool[4, :4].view(torch.int32).item()) == 0  # magic 0
    before, obs0, ram0 = _blobs(b), b.obs_tensor().clone(), b.ram_tensor().clone()
    slot_of = np.array([0, 1, 2, 6, 4, -1, 3, -7], np.int32)
    res = b.restore_states(pool, i32(slot_of)).cpu().numpy()
    assert res.tolist() == [2, 2, 2, 2, 2, 0, 1, 0]
    after = _blobs(b)
    untouched = res != 1
    assert np.array_equal(after[untouched], before[untouched])
    A = b.A
    img = torch.from_numpy(np.repeat(untouched, A)).cuda()
    assert torch.equal(b.obs_tensor()[img], obs0[img])
    assert torch.equal(b.ram_tensor()[torch.from_numpy(untouched).cuda()], ram0[torch.from_numpy(untouched).cuda()])
    assert np.array_equal(after[6], before[0])
    # the same pool into a batch of the same configuration with another n_instances and instance_base
    c = Batch(make_cfg(n_instances=5, instance_base=100, ram_obs=1, **SMALL))
    c.seed(8)
    c.reset()
    res = c.restore_states(pool, i32([3, -1, -1, 0, 3])).cpu().numpy()
    assert res.tolist() == [1, 0, 0, 2, 1]
    cb = _blobs(c)
    assert np.array_equal(cb[0], before[0]) and np.array_equal(cb[4], before[0])
    assert torch.equal(c.ram_tensor()[0], ram0[0])
    b.close()
    c.close()


@pytest.mark.gpu
def test_refusals_before_anything_is_enqueued():
    import torch
    from agarcl_b200._lib import AgarclError, lib
    from agarcl_b200.batch import Batch
    N = 4
    b = Batch(make_cfg(n_instances=N, **SMALL))
    pool = b.snapshot_pool(N)
    idx = i32(np.arange(N))
    with pytest.raises(AgarclError, match="before reset"):
        b.restore_states(pool, idx)
    with pytest.raises(AgarclError, match="before reset"):
        b.save_states(pool, idx)
    b.seed(5)
    b.reset()
    rng = np.random.default_rng(6)
    for _ in range(3):
        b.set_actions(*_actions(rng, N))
        b.step()
    b.save_states(pool, idx)
    torch.cuda.synchronize()
    before, obs0 = _blobs(b), b.obs_tensor().clone()
    sb = b.slot_bytes
    flat = torch.zeros(N * sb + 16, dtype=torch.uint8, device="cuda")
    flat[1:1 + N * sb] = pool.view(-1)
    misaligned = flat[1:1 + N * sb].view(N, sb)
    with pytest.raises(AgarclError, match="16-byte aligned"):
        b.restore_states(misaligned, idx)
    with pytest.raises(AgarclError, match="16-byte aligned"):
        b.save_states(misaligned, idx)
    with pytest.raises(AgarclError, match="tensor on cuda"):
        b.restore_states(pool.cpu(), idx)
    with pytest.raises(AgarclError, match="uint8"):
        b.restore_states(pool.view(torch.int8), idx)
    with pytest.raises(AgarclError, match="int32"):
        b.restore_states(pool, idx.long())
    with pytest.raises(AgarclError, match="4 entries"):
        b.restore_states(pool, i32(np.arange(N + 1)))
    with pytest.raises(AgarclError, match=str(sb)):
        b.restore_states(pool[:, :sb - 128].contiguous(), idx)
    # the C ABI itself: host memory, pool_slots < 1, n < 0, null index arrays
    host = np.zeros(N * sb + 64, np.uint8)
    hp = (host.ctypes.data + 15) // 16 * 16
    L, vp, res = lib(), C.c_void_p, C.c_void_p()
    assert L.agarcl_batch_restore_states(b._h, vp(hp), N, vp(idx.data_ptr()), C.byref(res), None) != 0
    assert "device memory" in L.agarcl_last_error().decode()
    assert L.agarcl_batch_save_states(b._h, vp(hp), N, vp(idx.data_ptr()), None, N, None) != 0
    assert L.agarcl_batch_restore_states(b._h, vp(pool.data_ptr()), 0, vp(idx.data_ptr()), C.byref(res), None) != 0
    assert L.agarcl_batch_save_states(b._h, vp(pool.data_ptr()), N, vp(idx.data_ptr()), None, -1, None) != 0
    assert L.agarcl_batch_save_states(b._h, vp(pool.data_ptr()), N, None, None, 2, None) != 0
    assert L.agarcl_batch_restore_states(b._h, vp(pool.data_ptr()), N, None, C.byref(res), None) != 0
    assert L.agarcl_batch_save_states(b._h, None, N, vp(idx.data_ptr()), None, N, None) != 0
    torch.cuda.synchronize()
    assert np.array_equal(_blobs(b), before) and torch.equal(b.obs_tensor(), obs0)
    b.close()
    for kw, frag in ((dict(strict_reference=1, ticks_per_step=1), "strict_reference"),
                     (dict(rng_mode=RNG_MT19937, cap_replay=4096), "MT19937")):
        x = Batch(make_cfg(n_instances=N, **kw, **SMALL))
        x.seed(5)
        x.reset()
        torch.cuda.synchronize()
        xb = _blobs(x)
        xp = x.snapshot_pool(N)
        with pytest.raises(AgarclError, match=frag):
            x.save_states(xp, idx)
        with pytest.raises(AgarclError, match=frag):
            x.restore_states(xp, idx)
        torch.cuda.synchronize()
        assert np.array_equal(_blobs(x), xb) and not bool(xp.any())
        x.close()


@pytest.mark.gpu
def test_save_and_restore_do_not_wait_for_the_device():
    import torch
    from agarcl_b200.env import BatchedGridEnvironment
    N = 64
    env = BatchedGridEnvironment(N, num_bots=2, arena_size=200, num_pellets=100, num_viruses=2)
    env.seed(1)
    env.reset()
    pool = env.snapshot_pool(N)
    idx = i32(np.arange(N))
    s = torch.cuda.Stream()
    for _ in range(2):  # every kernel on the path is loaded before the timed calls
        env.save_states(pool, idx, stream=s.cuda_stream)
        env.restore_states(pool, idx, stream=s.cuda_stream)

    def calls():
        env.save_states(pool, idx, stream=s.cuda_stream)
        env.restore_states(pool, idx, stream=s.cuda_stream)

    assert_no_host_wait(calls, s)
    env.close()


def _stepped(cfg, steps, seed=12):
    from agarcl_b200.batch import Batch
    b = Batch(cfg)
    b.seed(seed)
    b.reset()
    rng = np.random.default_rng(seed)
    for _ in range(steps):
        b.set_actions(*_actions(rng, b.N * b.A))
        b.step()
    return b


@pytest.mark.gpu
def test_pool_survives_torch_save_and_load():
    import torch
    from agarcl_b200.batch import Batch
    N = 6
    cfg = make_cfg(n_instances=N, num_frames=2, ram_obs=1, **SMALL)
    b = _stepped(cfg, 8)
    pool = b.snapshot_pool(N)
    b.save_states(pool, i32(np.arange(N)))
    buf = io.BytesIO()
    torch.save(pool.cpu(), buf)
    buf.seek(0)
    loaded = torch.load(buf).cuda()
    c = Batch(cfg)
    c.seed(77)
    c.reset()
    res = c.restore_states(loaded, i32(np.arange(N)[::-1].copy()))
    assert (res.cpu().numpy() == 1).all()
    assert np.array_equal(_blobs(c), _blobs(b)[::-1])
    A = b.A
    assert torch.equal(c.obs_tensor().view(N, A, -1).flip(0), b.obs_tensor().view(N, A, -1))
    assert torch.equal(c.ram_tensor().flip(0), b.ram_tensor())
    b.close()
    c.close()


@pytest.mark.gpu
def test_pool_moved_to_another_device():
    import torch
    from agarcl_b200.batch import Batch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    N = 4
    b = _stepped(make_cfg(n_instances=N, **SMALL), 6)
    pool = b.snapshot_pool(N)
    b.save_states(pool, i32(np.arange(N)))
    c = Batch(make_cfg(n_instances=N, device=1, **SMALL))
    c.seed(1)
    c.reset()
    res = c.restore_states(pool.to("cuda:1"), torch.arange(N, dtype=torch.int32, device="cuda:1"))
    assert (res.cpu().numpy() == 1).all()
    assert np.array_equal(_blobs(c), _blobs(b))
    assert torch.equal(c.obs_tensor().cpu(), b.obs_tensor().cpu())
    b.close()
    c.close()


@pytest.mark.gpu
def test_mirror_after_restore():
    import torch
    from agarcl_b200.batch import Batch
    N = 8
    b = Batch(make_cfg(n_instances=N, **SMALL))
    b.seed(2)
    b.reset()
    rng = np.random.default_rng(2)
    pool = b.snapshot_pool(N)
    for t in range(12):
        b.step_mirror(*_actions(rng, N))
        if t == 4:
            b.save_states(pool, i32(np.arange(N)))
    b.restore_states(pool, i32([0, -1, 2, 2, -1, 5, 6, 0]))
    m = b.sync_mirror()
    assert np.array_equal(m, b.obs_tensor().cpu().numpy())
    for _ in range(3):
        m = b.step_mirror(*_actions(rng, N))
        torch.cuda.synchronize()
        assert np.array_equal(m, b.obs_tensor().cpu().numpy())
    b.close()


@pytest.mark.gpu
def test_vector_env_restore():
    """BatchedAgarioEnv.restore_states returns the restored observation; a restored episode ends at the same length as one that
    was never restored: an instance restored at step s of a number_steps = 37 episode resets 37 - s steps later, plus the step on
    which the limit is checked (episode length 38, like any)"""
    import torch
    from agarcl_b200.gym_env import BatchedAgarioEnv
    N, limit, s = 8, 37, 10
    env = BatchedAgarioEnv(N, num_bots=0, arena_size=300, num_pellets=200, num_viruses=0, number_steps=limit)
    env.seed(4)
    env.reset()
    zeros = lambda: (torch.rand((N, 2), device="cuda") * 2 - 1, torch.zeros(N, dtype=torch.int32, device="cuda"))  # noqa: E731
    for _ in range(s):
        obs, _, _, _, info = env.step(*zeros())
    assert bool((info["steps"] == s).all())
    pool = env.snapshot_pool(N)
    env.save_states(pool, i32(np.arange(N)))
    saved = obs.clone()
    for _ in range(5):
        env.step(*zeros())
    obs = env.restore_states(pool, i32(np.arange(N)))
    assert torch.equal(obs, saved)
    assert (env.restore_result().cpu().numpy() == 1).all()
    assert bool((env._env.episode()["steps"] == s).all())
    for k in range(1, limit - s + 2):
        _, _, done, _, info = env.step(*zeros())
        ended = k == limit - s + 1
        assert bool(info["reset_mask"].all()) == ended and bool(info["reset_mask"].any()) == ended, k
        if ended:
            assert bool((info["episode_length"] == limit + 1).all())
    env.close()


LAUNCH_CASES = {"configs1": (dict(), ["k_obs", "k_snapshot"]), "int16": (CASES["int16"][0], ["k_obs", "k_snapshot"]),
                "two_frames": (CASES["two_frames"][0], ["k_snapshot"]), "ram_obs1": (CASES["ram_obs1"][0], ["k_obs", "k_snapshot"]),
                "ram_obs2": (CASES["ram_obs2"][0], ["k_snapshot"])}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LAUNCH_CASES))
def test_launches_of_a_restore(name):
    """a restore is k_snapshot, plus k_obs for a one-frame grid observation; a save is one k_snapshot"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    kw, want = LAUNCH_CASES[name]
    N = 8
    b = _stepped(make_cfg(n_instances=N, **kw), 2)
    pool = b.snapshot_pool(N)
    idx = i32(np.arange(N))
    torch.cuda.synchronize()

    def kernels(fn):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events()
                 if e.device_type == torch.autograd.DeviceType.CUDA and "Activity Buffer" not in e.name]
        return sorted(next((k for k in ("k_snapshot", "k_obs") if k in n), n) for n in names)

    assert kernels(lambda: b.save_states(pool, idx)) == ["k_snapshot"]
    assert kernels(lambda: b.restore_states(pool, idx)) == want
    b.close()
