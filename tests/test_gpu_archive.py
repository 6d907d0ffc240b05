"""The Go-Explore cell archive on the device (agarcl_batch_set_archive, archive_kernel.cu) against its numpy model
(archive_model.py) after every step: every array and counter, and every byte of the pool.  The model reads the games as they
are after the step and before any reset from a twin batch that is restored to the archive batch's games before every step and
then stepped alike (restore_states keys the draws by the same global index and cursor, so the twin's step is the same step).
Also: bit-identity with twins without an archive (select = 0) and with the model's picks as a start-state table (select = 1),
contention of forks, the pool's boundaries, refusals, host waits, graph capture and the step's launches."""
import numpy as np
import pytest

from agarcl_b200 import BOT_HUNGRY, OBS_I16, RNG_MT19937, make_cfg
from agarcl_b200._abi import StateView
from archive_model import ArchiveModel
from gpu_parity_lib import CASES, SMALL, assert_no_host_wait, device_record, i32

ARCHIVE_SEED = (0x1234 << 32) | 0x42
# name: (make_cfg keywords, cells_per_side, agent, episode limit, entries)
MODEL_CASES = {
    "configs1": (dict(), 8, 0, 60, 48),
    "small": (SMALL, 8, 0, 40, 48),
    "mode9_deaths_and_limit": (CASES["mode9_deaths_and_limit"][0], 8, 0, 37, 48),
    "two_agents_agent1": (dict(num_agents=2, **SMALL), 8, 1, 40, 48),
    "int16": (dict(obs_dtype=OBS_I16, **SMALL), 8, 0, 40, 48),
    "ram_obs1": (dict(ram_obs=1, **SMALL), 8, 0, 40, 48),
    "two_frames": (dict(num_frames=2, **SMALL), 8, 0, 40, 48),
    "pixels": (dict(pixel_obs=32, **SMALL), 8, 0, 40, 48),
    "n1": (SMALL, 1, 0, 40, 48),
    "n64": (SMALL, 64, 0, 40, 48),
    "full_archive": (SMALL, 16, 0, 40, 8),
}


def _random(rng, n):
    return rng.uniform(-1, 1, size=(n, 2)).astype(np.float32), rng.integers(0, 3, size=n).astype(np.int32)


def _run(kw, n, agent, limit, K, steps=300, N=8, select=True, twin=None, fork=False, seed=11):
    """steps step_autoresets of a batch with an archive, checked against the model after every one; with twin "plain" (select =
    0) or "table" (select = 1) a third batch is stepped alike and must hold exactly the same games.  Halfway, an explicit
    reset_device of every other instance.  Returns the archive's read-out and pool on the host."""
    import torch
    from agarcl_b200.batch import Batch
    cfg = make_cfg(n_instances=N, **kw)
    x, y = Batch(cfg), Batch(cfg)
    z = Batch(cfg) if twin else None
    bs = [b for b in (x, y, z) if b is not None]
    for b in bs:
        b.seed(seed)
        b.reset()
    A, L, sb = x.A, x.layout, x.slot_bytes
    every = i32(np.arange(N))
    sync, chk = x.snapshot_pool(N), x.snapshot_pool(N)
    rng = np.random.default_rng(seed)
    if fork:  # every instance begins in the game of instance 0 after a few steps
        for _ in range(4):
            for b in bs:
                b.set_actions(*_random(np.random.default_rng(1), N * A))
                b.step()
        x.save_states(sync, i32([0]))
        for b in bs:
            b.restore_states(sync, i32(np.zeros(N)))
    for b in (x, z):
        if b is not None:
            b.set_autoreset(limit)
    pool = x.snapshot_pool(K)
    x.set_archive(pool, n, agent=agent, select=select, seed=ARCHIVE_SEED)
    zpool = z.snapshot_pool(K) if twin == "table" else None
    model = ArchiveModel(N, A, K, n, agent, float(cfg.arena_size), seed=ARCHIVE_SEED, instance_base=cfg.instance_base, select=select)
    off_ep = 64 + L.stride
    host_pool = np.zeros((K, sb), np.uint8)
    ret = np.zeros(N * A)
    ep = x.episode()
    resets = 0

    def after_reset(mask):
        nonlocal ret
        picks = model.select(mask)
        res = x.start_result().cpu().numpy()
        if select:
            want = np.array([1 if mask[i] and picks.get(i, -1) >= 0 else 0 for i in range(N)], np.uint8)
            assert np.array_equal(res, want), (res, want)
        model.set_base(mask, {i: e for i, e in picks.items() if e >= 0 and res[i] == 1})
        ret = np.where(np.repeat(mask, A), 0.0, ret)
        return picks

    def twin_reset(picks, call):
        if twin == "table":
            zpool.copy_(pool)
            z.set_start_states(zpool, i32([picks.get(i, -1) for i in range(N)]))
        call(z)

    for t in range(steps):
        steps_before = ep["steps"].cpu().numpy().copy()
        x.save_states(sync, every)
        y.restore_states(sync, every)
        if t % 2 and not fork:
            dxdy, act, _ = x.bot_actions(BOT_HUNGRY)
            for b in (y, x, z):
                if b is not None:
                    b.set_actions_device(dxdy.data_ptr(), act.data_ptr())
        else:
            acts = _random(rng, A) if fork else _random(rng, N * A)
            acts = (np.tile(acts[0], (N, 1)), np.tile(acts[1], N)) if fork else acts
            for b in bs:
                b.set_actions(*acts)
        y.step()
        x.step_autoreset()
        y.save_states(chk, every)
        torch.cuda.synchronize()
        c = chk.cpu().numpy()
        rew = y.rewards_tensor().cpu().numpy()
        saves = model.update([StateView(L, c[i, 64:64 + L.stride].copy()) for i in range(N)], y.dones_tensor().cpu().numpy(), rew,
                             ret, steps_before)
        for e, i in saves.items():  # what save_states writes at that moment: the episode record before the bookkeeping
            host_pool[e] = c[i]
            host_pool[e, off_ep:off_ep + 8] = np.array([steps_before[i]], np.int64).view(np.uint8)
            host_pool[e, off_ep + 8:off_ep + 8 + 8 * A] = ret[i * A:(i + 1) * A].astype(np.float64).view(np.uint8)
        ret = ret + rew
        mask = ep["reset_mask"].cpu().numpy().astype(bool)
        resets += int(mask.sum())
        picks = after_reset(mask)
        if z is not None:
            twin_reset(picks, lambda b: b.step_autoreset())
        if t == steps // 2:  # an explicit reset of every other instance
            m = (np.arange(N) % 2 == 0).astype(np.uint8)
            x.reset_device(i32(m).to(torch.uint8))
            torch.cuda.synchronize()
            picks = after_reset(m.astype(bool))
            if z is not None:
                twin_reset(picks, lambda b: b.reset_device(i32(m).to(torch.uint8)))
        got = {k: v.cpu().numpy() for k, v in x.archive().items()}
        for k, v in model.arrays().items():
            assert np.array_equal(got[k], v), f"step {t}: {k}"
        assert np.array_equal(pool.cpu().numpy(), host_pool), f"step {t}: pool"
        if z is not None:
            rx, rz = device_record(x), device_record(z)
            for k in rx:
                assert np.array_equal(rx[k], rz[k]), f"step {t}: twin {k}"
    assert resets >= N // 2, resets  # (forks with one action sequence reset together: the explicit reset splits them in two)
    out = {k: v.cpu().numpy() for k, v in x.archive().items()}, pool.cpu().numpy()
    for b in bs:
        b.close()
    return out, model


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODEL_CASES))
def test_archive_equals_the_model(name):
    (arch, _), model = _run(*MODEL_CASES[name])
    assert model.used > 1 and arch["counters"][0] == model.used
    if name == "full_archive":
        assert model.dropped > 0 and model.used == 8
    if name == "n1":
        assert model.used <= 32


@pytest.mark.gpu
@pytest.mark.parametrize("select,twin", [(False, "plain"), (True, "table")])
def test_games_equal_a_twin(select, twin):
    """select = 0: the games are bit-identical to a batch without an archive; select = 1: to a batch whose start-state table is
    set every step to the model's picks on a copy of the pool"""
    _run(SMALL, 8, 0, 25, 32, steps=150, select=select, twin=twin)


@pytest.mark.gpu
def test_contention_of_forks():
    """forks of one game with identical actions fight over the same cells: the model holds, and two runs give identical archives"""
    _run(SMALL, 8, 0, 25, 32, steps=100, N=64, fork=True)
    runs = [_run(SMALL, 8, 0, 25, 64, steps=40, N=256, fork=True, seed=5)[0] for _ in range(2)]
    for k in runs[0][0]:
        assert np.array_equal(runs[0][0][k], runs[1][0][k]), k
    assert np.array_equal(runs[0][1], runs[1][1])
    assert runs[0][0]["visits"].sum() > 256


@pytest.mark.gpu
def test_pool_boundaries():
    """K = 8 inside a larger buffer: discoveries beyond 8 are dropped and nothing is written outside the 8 slots"""
    import torch
    from agarcl_b200.batch import Batch
    N = 32
    b = Batch(make_cfg(n_instances=N, **SMALL))
    b.seed(3)
    b.reset()
    b.set_autoreset(30)
    buf = torch.full((10, b.slot_bytes), 0xAB, dtype=torch.uint8, device="cuda")
    b.set_archive(buf[1:9], 16)
    rng = np.random.default_rng(3)
    for _ in range(80):
        b.set_actions(*_random(rng, N * b.A))
        b.step_autoreset()
    a = {k: v.cpu().numpy() for k, v in b.archive().items()}
    used, dropped, _ = a["counters"].tolist()
    assert used == 8 and dropped > 0
    assert (buf[0] == 0xAB).all() and (buf[9] == 0xAB).all()
    assert sorted(a["entry_key"].tolist()) == sorted(np.flatnonzero(a["key_entry"] >= 0).tolist())
    b.close()


@pytest.mark.gpu
def test_refusals_leave_the_archive():
    import ctypes as C
    import torch
    from agarcl_b200._abi import ArchiveCfg
    from agarcl_b200._lib import AgarclError, lib
    from agarcl_b200.batch import Batch
    N = 4
    b = Batch(make_cfg(n_instances=N, **SMALL))
    b.seed(1)
    b.reset()
    pool = b.snapshot_pool(8)
    with pytest.raises(AgarclError, match="set_autoreset"):
        b.set_archive(pool, 8)
    b.set_autoreset(20, reset=False)
    with pytest.raises(AgarclError, match="set_autoreset"):
        b.set_archive(pool, 8)
    b.set_autoreset(20)
    b.set_archive(pool, 8)
    rng = np.random.default_rng(1)
    for _ in range(6):
        b.set_actions(*_random(rng, N))
        b.step_autoreset()
    before = {k: v.cpu().numpy() for k, v in b.archive().items()}
    for kw, frag in ((dict(cells_per_side=0), "cells_per_side"), (dict(cells_per_side=257), "cells_per_side"),
                     (dict(cells_per_side=8, agent=1), "agent"), (dict(cells_per_side=8, agent=-1), "agent")):
        with pytest.raises(AgarclError, match=frag):
            b.set_archive(pool, **kw)
    flat = torch.zeros(8 * b.slot_bytes + 16, dtype=torch.uint8, device="cuda")
    with pytest.raises(AgarclError, match="16-byte aligned"):
        b.set_archive(flat[1:1 + 8 * b.slot_bytes].view(8, b.slot_bytes), 8)
    L, vp = lib(), C.c_void_p
    cfg = ArchiveCfg(cells_per_side=8, agent=0, select=1, pad=0, seed=0)
    host = np.zeros(8 * b.slot_bytes + 64, np.uint8)
    assert L.agarcl_batch_set_archive(b._h, vp((host.ctypes.data + 15) // 16 * 16), 8, C.byref(cfg)) != 0
    assert "device memory" in L.agarcl_last_error().decode()
    assert L.agarcl_batch_set_archive(b._h, vp(pool.data_ptr()), 0, C.byref(cfg)) != 0
    assert L.agarcl_batch_set_archive(b._h, vp(pool.data_ptr()), 65537, C.byref(cfg)) != 0
    cfg.select = 2
    assert L.agarcl_batch_set_archive(b._h, vp(pool.data_ptr()), 8, C.byref(cfg)) != 0
    with pytest.raises(AgarclError, match="owns the start-state table"):
        b.set_start_states(pool, i32(np.zeros(N)))
    with pytest.raises(AgarclError, match="archive"):
        b.set_autoreset(20, reset=False)
    after = {k: v.cpu().numpy() for k, v in b.archive().items()}
    for k in before:
        assert np.array_equal(before[k], after[k]), k
    b.set_archive(None)
    assert b._start_pool is None
    with pytest.raises(AgarclError, match="no archive"):
        b.archive()
    b.set_start_states(None)  # the table is the caller's again
    b.close()
    for kw, frag in ((dict(strict_reference=1, ticks_per_step=1, **SMALL), "strict_reference"),
                     (dict(rng_mode=RNG_MT19937, cap_replay=4096, **SMALL), "MT19937"), (CASES["mixed_tasks"][0], "mixed-task")):
        x = Batch(make_cfg(n_instances=N, **kw))
        x.set_autoreset(10)
        with pytest.raises(AgarclError, match=frag):
            x.set_archive(x.snapshot_pool(4), 8)
        x.close()


@pytest.mark.gpu
def test_restore_clears_the_base():
    import torch
    from agarcl_b200.batch import Batch
    N = 8
    b = Batch(make_cfg(n_instances=N, **dict(SMALL, num_bots=0)))
    b.seed(2)
    b.reset()
    b.set_autoreset(5)
    b.set_archive(b.snapshot_pool(32), 8)
    rng = np.random.default_rng(2)
    for _ in range(12):  # every instance has restarted from an entry: bases > 0 where the entry had a positive score
        b.set_actions(*_random(rng, N))
        b.step_autoreset()
    torch.cuda.synchronize()
    base = b.archive()["base_length"].cpu().numpy().copy()
    assert (base > 0).all(), base
    p = b.snapshot_pool(N)
    b.save_states(p, i32(np.arange(N)))
    b.restore_states(p, i32([0, -1, 2, -1, -1, -1, -1, -1]))
    after = b.archive()["base_length"].cpu().numpy()
    assert after[0] == 0 and after[2] == 0 and np.array_equal(np.delete(after, [0, 2]), np.delete(base, [0, 2]))
    b.close()


@pytest.mark.gpu
def test_no_host_wait_graph_capture_and_launches():
    import torch
    from agarcl_b200.batch import Batch
    from agarcl_b200.env import BatchedGridEnvironment
    M = 64
    env = BatchedGridEnvironment(M, num_bots=2, arena_size=200, num_pellets=100, num_viruses=2)
    env.seed(1)
    env.reset()
    env.set_autoreset(3)
    pool = env.snapshot_pool(64)
    env.set_archive(pool, 8)
    s = torch.cuda.Stream()
    dxdy, act = torch.zeros((M, 2), device="cuda"), torch.zeros(M, dtype=torch.int32, device="cuda")
    mask, every = i32(np.arange(M) % 2).to(torch.uint8), i32(np.arange(M))
    for _ in range(4):
        env.step_autoreset(dxdy, act, stream=s.cuda_stream)
    env.batch.reset_device(mask, stream=s.cuda_stream)
    env.save_states(pool, every, stream=s.cuda_stream)
    env.restore_states(pool, every, stream=s.cuda_stream)

    def calls():
        for _ in range(3):
            env.step_autoreset(dxdy, act, stream=s.cuda_stream)
        env.batch.reset_device(mask, stream=s.cuda_stream)
        env.restore_states(pool, every, stream=s.cuda_stream)

    assert_no_host_wait(calls, s)
    env.close()
    # the step's launches do not change with an archive
    N = 8
    cfg = make_cfg(n_instances=N, **SMALL)
    plain, arch = Batch(cfg), Batch(cfg)
    for b in (plain, arch):
        b.seed(4)
        b.reset()
        b.set_autoreset(6)
    arch.set_archive(arch.snapshot_pool(16), 8)
    acts = _random(np.random.default_rng(4), N)
    for b in (plain, arch):
        b.set_actions(*acts)
        b.step_autoreset()
    assert plain.launches_per_step() == arch.launches_per_step()
    # a CUDA graph of step_autoreset, if one can be captured without an archive, can be captured with one and replays alike
    d = (torch.tensor(acts[0], device="cuda"), torch.tensor(acts[1], device="cuda"))
    g = torch.cuda.CUDAGraph()
    for b in (plain, arch):
        b.set_actions_device(d[0].data_ptr(), d[1].data_ptr())
    try:
        with torch.cuda.graph(torch.cuda.CUDAGraph(), stream=s):
            plain.step_autoreset(stream=s.cuda_stream)
    except Exception as e:  # noqa: BLE001
        pytest.skip(f"step_autoreset cannot be captured without an archive either: {e}")
    twin = Batch(cfg)
    twin.seed(4)
    twin.reset()
    twin.set_autoreset(6)
    twin.set_archive(twin.snapshot_pool(16), 8)
    twin.set_actions(*acts)
    twin.step_autoreset()
    twin.set_actions_device(d[0].data_ptr(), d[1].data_ptr())
    with torch.cuda.graph(g, stream=s):
        arch.step_autoreset(stream=s.cuda_stream)
    for _ in range(10):
        g.replay()
        twin.step_autoreset()
    torch.cuda.synchronize()
    ra, rt = device_record(arch), device_record(twin)
    for k in ra:
        assert np.array_equal(ra[k], rt[k]), k
    aa, at = arch.archive(), twin.archive()
    for k in aa:
        assert np.array_equal(aa[k].cpu().numpy(), at[k].cpu().numpy()), k
    for b in (plain, arch, twin):
        b.close()


@pytest.mark.gpu
def test_vector_env_archive():
    import torch
    from agarcl_b200.gym_env import BatchedAgarioEnv
    N = 16
    env = BatchedAgarioEnv(N, num_bots=0, arena_size=200, num_pellets=100, num_viruses=2, number_steps=6)
    env.seed(3)
    env.reset()
    env.set_archive(64, cells_per_side=8, seed=9)
    g = torch.Generator(device="cuda").manual_seed(3)
    for _ in range(20):
        dxdy = torch.rand((N, 2), device="cuda", generator=g) * 2 - 1
        _, _, _, _, info = env.step(dxdy, torch.zeros(N, dtype=torch.int32, device="cuda"))
        assert torch.equal(info["cell"], env.archive()["cell_of"]) and "start_result" in info
    a = {k: v.cpu().numpy() for k, v in env.archive().items()}
    assert a["counters"][0] > 1 and a["entry_chosen"].sum() > 0
    env.set_archive(None)
    _, _, _, _, info = env.step(dxdy, torch.zeros(N, dtype=torch.int32, device="cuda"))
    assert "cell" not in info and "start_result" not in info
    env.close()
