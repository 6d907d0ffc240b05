"""Auto-reset on the device (agarcl_batch_step_autoreset, agarcl_batch_reset_device): equal, bit for bit, to the composition
it replaces -- step, the reset mask computed on the host from the downloaded dones and a host step counter, then
agarcl_batch_reset with that host mask -- and the host never waits for the device on its way."""
import ctypes as C

import numpy as np
import pytest

from agarcl_b200 import OBS_I16, make_cfg
from gpu_parity_lib import CASES, assert_no_host_wait, device_record


def test_episode_struct_matches_header():
    from agarcl_b200.batch import _EpisodeStruct
    assert C.sizeof(_EpisodeStruct) == 7 * 8  # struct agarcl_episode: seven pointers
    assert [f[0] for f in _EpisodeStruct._fields_] == ["done_out", "reset_mask", "steps", "final_return", "final_length",
                                                       "final_obs", "final_ram"]


def _pair(cfg, seed):
    from agarcl_b200.batch import Batch
    ref, dev = Batch(cfg), Batch(cfg)
    for b in (ref, dev):
        b.seed(seed)
        b.reset()
    return ref, dev


AUTORESET_CASES = ["mode9_deaths_and_limit", "configs1_two_agents", "int16", "two_frames", "strict_reference", "ram_obs1", "ram_obs2",
                   "mt19937_ring_wraps"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", AUTORESET_CASES)
def test_step_autoreset_equals_host_composition(name):
    import torch
    kw = CASES[name][0]
    N, steps, max_steps = (16 if name == "configs1_two_agents" else 32), 200, 37
    cfg = make_cfg(n_instances=N, **kw)
    ref, dev = _pair(cfg, 1234)
    A, grid = ref.A, cfg.ram_obs != 2
    dev.set_autoreset(max_steps, keep_final_obs=True)
    ep = dev.episode()
    final_obs = dev.final_obs() if grid else None
    final_ram = dev.final_ram() if cfg.ram_obs else None
    if not grid:
        with pytest.raises(RuntimeError):
            dev.final_obs()
    host_steps = np.zeros(N, np.int64)
    acc = np.zeros(N * A, np.float64)
    rng = np.random.default_rng(7)
    deaths = truncations = 0
    for t in range(steps):
        dxdy = rng.uniform(-1, 1, size=(N * A, 2)).astype(np.float32)
        act = rng.integers(0, 3, size=N * A).astype(np.int32)
        # the reference composition (what BatchedAgarioEnv did on the host)
        ref.set_actions(dxdy, act)
        ref.step()
        dones = ref.dones_tensor().cpu().numpy().astype(bool).reshape(N, A)
        rew = ref.rewards_tensor().cpu().numpy()
        limit = host_steps >= max_steps
        done = dones | limit[:, None]
        host_steps += 1
        acc += rew
        mask = done.any(axis=1)
        deaths += int((dones.any(axis=1) & ~limit).sum())
        truncations += int((limit & ~dones.any(axis=1)).sum())
        pre_obs = ref.obs_tensor().clone() if grid else None
        pre_ram = ref.ram_tensor().clone() if cfg.ram_obs else None
        if mask.any():
            ref.reset(mask.astype(np.uint8))
        # the device path
        dev.set_actions(dxdy, act)
        dev.step_autoreset()
        torch.cuda.synchronize()
        img = torch.from_numpy(np.repeat(mask, A)).cuda()
        r, d = device_record(ref), device_record(dev)
        for k in r:  # state blobs, obs, rewards, dones and ram records
            assert np.array_equal(r[k], d[k]), (t, k)
        assert np.array_equal(ep["done"].cpu().numpy(), done.reshape(-1).astype(np.uint8)), t
        assert np.array_equal(ep["reset_mask"].cpu().numpy(), mask.astype(np.uint8)), t
        if mask.any():
            agents = np.repeat(mask, A)
            assert np.array_equal(ep["episode_return"].cpu().numpy()[agents], acc[agents]), t
            assert np.array_equal(ep["episode_length"].cpu().numpy()[mask], host_steps[mask]), t
            if grid:
                assert torch.equal(final_obs[img], pre_obs[img]), t
            if cfg.ram_obs:
                m = torch.from_numpy(mask).cuda()
                assert torch.equal(final_ram[m], pre_ram[m]), t
            acc[agents] = 0.0
            host_steps[mask] = 0
        assert np.array_equal(ep["steps"].cpu().numpy(), host_steps), t
    assert truncations > 0
    if name == "mode9_deaths_and_limit":
        assert deaths > 0, "no agent died: the run did not cover natural episode ends"
    if name == "mt19937_ring_wraps":
        assert min(int(dev.download_state(i).hdr["rng_cursor"]) for i in range(N)) > 2 * 1024
        assert not (dev.flags()[0] & 0x20)  # never AGARCL_FLAG_REPLAY_EXHAUSTED
    ref.close()
    dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(num_bots=4, arena_size=300, num_pellets=300, num_viruses=4),
                                # per-instance observation of 26136 bytes and ram records: heads and tails off 16-byte bounds
                                dict(num_frames=2, grid_size=33, observe_others=False, obs_dtype=OBS_I16, ram_obs=1, num_bots=4,
                                     arena_size=300, num_pellets=300, num_viruses=4)])
def test_device_mask_reset(kw):
    """reset(CUDA mask) == reset(host mask); the instances it resets equal those of a full reset (cleared with memsets), and
    the others keep their state, observation and ram records"""
    import torch
    from agarcl_b200.batch import Batch
    N = 24
    cfg = make_cfg(n_instances=N, **kw)
    bs = [Batch(cfg) for _ in range(3)]
    rng = np.random.default_rng(3)
    for b in bs:
        b.seed(55)
        b.reset()
    for _ in range(20):
        dxdy = rng.uniform(-1, 1, size=(N, 2)).astype(np.float32)
        act = rng.integers(0, 3, size=N).astype(np.int32)
        for b in bs:
            b.set_actions(dxdy, act)
            b.step()
    mask = (rng.random(N) < 0.4).astype(np.uint8)
    mask[0], mask[1] = 1, 0
    before = [bs[1].download_state(i).blob.copy() for i in range(N)]
    obs_before = bs[1].obs_tensor().clone()
    ram_before = bs[1].ram_tensor().clone() if cfg.ram_obs else None
    bs[0].reset(mask)
    bs[1].reset_device(torch.from_numpy(mask).cuda().bool())
    bs[2].reset()
    r0, r1 = device_record(bs[0]), device_record(bs[1])
    for k in r0:
        assert np.array_equal(r0[k], r1[k]), k
    img = torch.from_numpy(np.repeat(mask.astype(bool), bs[1].A)).cuda()
    m = torch.from_numpy(mask.astype(bool)).cuda()
    o1, o2 = bs[1].obs_tensor(), bs[2].obs_tensor()
    assert torch.equal(o1[img], o2[img]) and torch.equal(o1[~img], obs_before[~img])
    if cfg.ram_obs:
        r1 = bs[1].ram_tensor()
        assert int(r1[m].abs().sum()) == 0 and torch.equal(r1[~m], ram_before[~m])
    for i in range(N):
        if mask[i]:
            assert np.array_equal(bs[1].download_state(i).blob, bs[2].download_state(i).blob), i
        else:
            assert np.array_equal(bs[1].download_state(i).blob, before[i]), i
    for b in bs:
        b.close()


@pytest.mark.gpu
def test_step_autoreset_does_not_wait_for_the_device():
    """The host returns from every call while the stream is still busy with work queued before them.  (Detects a
    synchronise on the way; the device only sleeps.)"""
    import torch
    from agarcl_b200.env import BatchedGridEnvironment
    from agarcl_b200.gym_env import BatchedAgarioEnv
    N = 64
    env = BatchedGridEnvironment(N, num_bots=2, arena_size=200, num_pellets=100, num_viruses=2)
    env.seed(1)
    env.reset()
    env.set_autoreset(3, final_obs=True)
    s = torch.cuda.Stream()
    dxdy = torch.zeros((N, 2), device="cuda")
    act = torch.zeros(N, dtype=torch.int32, device="cuda")
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
    mask[::3] = 1
    for _ in range(4):  # every kernel on the path is loaded before the timed calls (and some instances reset)
        env.step_autoreset(dxdy, act, stream=s.cuda_stream)
        env.reset(mask, stream=s.cuda_stream)

    def calls():
        for _ in range(3):
            env.step_autoreset(dxdy, act, stream=s.cuda_stream)
        env.reset(mask, stream=s.cuda_stream)

    assert_no_host_wait(calls, s)
    steps = env.episode()["steps"].cpu().numpy()
    assert steps.max() <= 3 and (steps[::3] == 0).all()
    env.close()
    # the vector environment on the current stream
    venv = BatchedAgarioEnv(N, num_bots=2, arena_size=200, num_pellets=100, num_viruses=2, number_steps=2, final_obs=True)
    venv.seed(2)
    venv.reset()
    for _ in range(4):
        venv.step(dxdy, act)
    assert_no_host_wait(lambda: [venv.step(dxdy, act) for _ in range(3)], torch.cuda.current_stream())
    venv.close()


@pytest.mark.gpu
def test_errors():
    import torch
    from agarcl_b200._lib import AgarclError
    from agarcl_b200.env import BatchedGridEnvironment
    from agarcl_b200.gym_env import BatchedAgarioEnv
    N = 8
    env = BatchedGridEnvironment(N, num_bots=1, arena_size=100, num_pellets=50, num_viruses=0)
    env.reset()
    dxdy, act = torch.zeros((N, 2), device="cuda"), torch.zeros(N, dtype=torch.int32, device="cuda")
    with pytest.raises(RuntimeError, match="set_autoreset"):
        env.step_autoreset(dxdy, act)
    with pytest.raises(RuntimeError, match="set_autoreset"):
        env.episode()
    b = env.batch
    with pytest.raises(AgarclError, match="tensor on cuda"):
        b.reset_device(torch.zeros(N, dtype=torch.uint8))  # host memory
    with pytest.raises(AgarclError, match="uint8 or bool"):
        env.reset(torch.zeros(N, dtype=torch.int32, device="cuda"))
    with pytest.raises(AgarclError, match="8 entries"):
        env.reset(torch.zeros(N + 1, dtype=torch.uint8, device="cuda"))
    with pytest.raises(AgarclError, match="8 entries"):
        env.reset(torch.zeros((N, 2), dtype=torch.uint8, device="cuda")[:, 0])  # not contiguous
    env.set_autoreset(5)
    with pytest.raises(AgarclError, match="final observation"):
        b.final_obs()
    with pytest.raises(AgarclError, match="final ram"):
        b.final_ram()
    with pytest.raises(RuntimeError, match="needs reset"):
        env.set_autoreset(5, final_obs=True, reset=False)
    with pytest.raises(RuntimeError, match="max_steps"):
        env.set_autoreset(-1)
    env.step_autoreset(dxdy, act)
    env.close()
    with pytest.raises(ValueError):
        BatchedAgarioEnv(4, auto_reset=False, final_obs=True)


@pytest.mark.gpu
def test_vector_env_info():
    """BatchedAgarioEnv: info's episode statistics and final observation against the step counter and the rewards it returned;
    with auto_reset=False nothing is reset, the limit stays folded into dones and steps counts on"""
    import torch
    from agarcl_b200.gym_env import BatchedAgarioEnv
    N, limit = 16, 5
    kw = dict(num_bots=2, arena_size=150, num_pellets=80, num_viruses=2, number_steps=limit)
    env = BatchedAgarioEnv(N, final_obs=True, **kw)
    env.seed(11)
    env.reset()
    ret = torch.zeros(N, dtype=torch.float64, device="cuda")
    for t in range(13):
        dxdy = torch.rand((N, 2), device="cuda") * 2 - 1
        act = torch.zeros(N, dtype=torch.int32, device="cuda")
        obs, rew, done, trunc, info = env.step(dxdy, act)
        assert set(info) == {"steps", "reset_mask", "episode_return", "episode_length", "final_obs"}
        ret += env._env.batch.rewards_tensor()
        assert torch.equal(rew, env._env.batch.rewards_tensor().float())
        m = info["reset_mask"]
        assert torch.equal(m, done) and not bool(trunc.any())
        if t % (limit + 1) == limit:
            assert bool(m.all()) and bool((info["episode_length"] == limit + 1).all())
            assert torch.equal(info["episode_return"], ret)
            assert not torch.equal(info["final_obs"], obs)  # the episode's last frame, not the new episode's first
            ret.zero_()
        else:
            assert not bool(m.any())
    env.close()
    env = BatchedAgarioEnv(N, auto_reset=False, **kw)
    env.seed(11)
    env.reset()
    for t in range(8):
        _, _, done, _, info = env.step(torch.zeros((N, 2), device="cuda"), torch.zeros(N, dtype=torch.int32, device="cuda"))
        assert set(info) == {"steps"} and bool((info["steps"] == t + 1).all())
        assert bool(done.all()) == (t >= limit)
    env.close()
