"""CUDA path vs oracle port, step by step, on identical initial state and identical draws.

Everything discrete (counts, masses, timers, cooldowns, statistics, rewards, dones, flags) and
every fp32 field must be IDENTICAL: the oracle runs with trig_mode 1 (the same restatement of
glibc's atanf / sinf / cosf as the device, itself equal to libm: tests/test_trig_exact.py), all
other arithmetic is IEEE-exact on both sides.

Also the scaffolding the device-feature tests share: the configuration catalogue CASES, aged
batches, the record of everything a batch holds and the no-host-wait check.
"""
import numpy as np

from _helpers import Oracle, oracle_lib, oracle_layout, random_actions
from agarcl_b200 import OBS_I16, RNG_MT19937, RNG_REPLAY, make_cfg
from agarcl_b200._abi import compare_states, task_bits
from agarcl_b200.batch import Batch

SMALL = dict(num_bots=4, arena_size=300, num_pellets=300, num_viruses=4)
# name: (make_cfg keywords, p_feed, p_split, boost); each test module selects its cases by name
CASES = {
    "c1": (dict(num_viruses=0, num_bots=0), 1 / 3, 1 / 3, None),
    "c2": (dict(), 1 / 3, 1 / 3, None),
    "c3": (dict(num_bots=8, num_viruses=10), 0.0, 0.0, None),
    "c4_four_agents": (dict(num_agents=4, num_bots=8, cap_foods=2048), 0.3, 0.3, 1000),
    "c5": (dict(arena_size=2000, num_pellets=4000, num_viruses=50, cap_viruses=128), 1 / 3, 1 / 3, None),
    "configs1_two_agents": (dict(num_agents=2), 1 / 3, 1 / 3, None),
    "mode1": (dict(mode_number=1, num_bots=0), 1 / 3, 1 / 3, None),
    "mode7": (dict(mode_number=7), 1 / 3, 1 / 3, None),
    "mode8": (dict(mode_number=8), 1 / 3, 1 / 3, None),
    "mode9": (dict(mode_number=9), 1 / 3, 1 / 3, None),
    "mode10": (dict(mode_number=10), 1 / 3, 1 / 3, None),
    # mode 9: its one bot is the Aggressive type, which eats the random-walking agent in about one 37-step episode in ten (the
    # Hungry-Shy bot of mode 8 never does in the oracle over 64 seeds), so an episodic run sees deaths as well as step-limit
    # truncations
    "mode9_deaths_and_limit": (dict(mode_number=9, num_bots=1, arena_size=200, num_pellets=300, num_viruses=0), 1 / 3, 1 / 3,
                               None),
    "mixed_tasks": (dict(mode_number=1, task_modes=task_bits([1, 7, 8, 10]), num_bots=0, arena_size=400, num_pellets=400), 1 / 3,
                    1 / 3, None),
    "int16": (dict(obs_dtype=OBS_I16, **SMALL), 1 / 3, 1 / 3, None),
    "two_frames": (dict(num_frames=2, **SMALL), 1 / 3, 1 / 3, None),
    "ram_obs1": (dict(ram_obs=1, **SMALL), 1 / 3, 1 / 3, None),
    "ram_obs2": (dict(ram_obs=2, **SMALL), 1 / 3, 1 / 3, None),
    "mt19937": (dict(rng_mode=RNG_MT19937, **SMALL), 1 / 3, 1 / 3, None),
    # one step draws at most 2 * (150 + 2 + 4) = 312: a 1024-entry ring wraps within a few episodes
    "mt19937_ring_wraps": (dict(rng_mode=RNG_MT19937, cap_replay=1024, num_bots=3, arena_size=60, num_pellets=150, num_viruses=2),
                           1 / 3, 1 / 3, None),
    # one tick per step: the step renders its frame with k_obs
    "strict_reference": (dict(strict_reference=1, ticks_per_step=1, num_agents=2, **SMALL), 1 / 3, 1 / 3, None),
}


def i32(x):
    import torch
    return torch.as_tensor(np.asarray(x, np.int32), device="cuda")


def aged_batch(name, N=4, seed=5, second_reset=False):
    """a Batch of N instances of CASES[name] seeded with `seed` and reset, with the rng, p_feed and p_split for step_random.
    A mixed-task batch plays modes 1, 7, 8, 10, then 1.  second_reset: under strict_reference, a second unmasked reset (the
    player order of the reference's second episode).  A boost is the mass of the agents' first cell after the reset."""
    import torch
    kw, p_feed, p_split, boost = CASES[name]
    b = Batch(make_cfg(n_instances=N, **kw))
    b.seed(seed)
    if b.cfg.task_modes:
        b.set_tasks(i32([1, 7, 8, 10][:N] + [1] * max(0, N - 4)))
    b.reset()
    if second_reset and b.cfg.strict_reference:
        b.reset()
    if boost:
        for i in range(N):
            sv = b.download_state(i)
            for a in range(b.A):
                sv.cells[a][0]["mass"] = boost
            b.upload_state(i, sv)
    torch.cuda.synchronize()
    return b, np.random.default_rng(seed), p_feed, p_split


def step_random(b, rng, p_feed, p_split, k):
    for _ in range(k):
        b.set_actions(*random_actions(rng, b.N * b.A, p_feed, p_split))
        b.step()


def device_record(b):
    """everything batch b holds, on the host: state blobs, observation, rewards and dones; ram records (cfg.ram_obs), the
    episode buffers with the final observations and ram records (after set_autoreset) and the host mirror (once made)"""
    import torch
    torch.cuda.synchronize()
    r = {"blobs": np.stack([b.download_state(i).blob for i in range(b.N)]), "obs": b.obs_tensor().cpu().numpy(),
         "rewards": b.rewards_tensor().cpu().numpy(), "dones": b.dones_tensor().cpu().numpy()}
    if b.cfg.ram_obs:
        r["ram"] = b.ram_tensor().cpu().numpy()
    if hasattr(b, "_episode"):
        r.update({k: v.cpu().numpy() for k, v in b.episode().items()})
        e = b._episode_struct()
        if e.final_obs:
            r["final_obs"] = b.final_obs().cpu().numpy()
        if e.final_ram:
            r["final_ram"] = b.final_ram().cpu().numpy()
    if getattr(b, "_mirror", None) is not None:
        r["mirror"] = b.mirror().copy()
    return r


def assert_no_host_wait(calls, stream):
    """the host returns from calls() while `stream` is still busy with work queued before them (detects a synchronise on the
    way; the device only sleeps).  Every kernel on the path must have been loaded before, by a warm-up."""
    import torch
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        torch.cuda._sleep(200_000_000)  # ~0.1 s at the B200's clock
    calls()
    busy = not stream.query()
    torch.cuda.synchronize()
    assert busy, "a call waited for the device"


def philox4x32_10_np(counter, key):
    """Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11; Random123) on arrays of
    counters: counter = 4 uint32 words (arrays or scalars), key = 2 words.  Pinned against Random123's known-answer vectors
    in tests/test_philox_kat.py; the device's philox4x32_10 (device_math.cuh) is then pinned against THIS by the RNG_PHILOX
    parity runs."""
    c = [np.asarray(x, dtype=np.uint64) for x in counter]
    key = [np.uint64(key[0]), np.uint64(key[1])]
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    mask = np.uint64(0xffffffff)
    for _ in range(10):
        p0 = M0 * c[0]
        p1 = M1 * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & mask
        hi1, lo1 = p1 >> np.uint64(32), p1 & mask
        c = [(hi1 ^ c[1] ^ key[0]) & mask, lo1, (hi0 ^ c[3] ^ key[1]) & mask, lo0]
        key = [(key[0] + np.uint64(0x9E3779B9)) & mask, (key[1] + np.uint64(0xBB67AE85)) & mask]
    return c


def philox_uniform_np(seed, instance, k):
    """numpy restatement of device_math.cuh::philox_uniform for draw indices k (test-side only): draw k of global instance
    g under 64-bit seed s = word (k & 3) of philox(counter = (k >> 2, 0, g, 0), key = (s_lo, s_hi)), top 24 bits -> [0, 1)."""
    k = np.asarray(k, dtype=np.uint64)
    c = philox4x32_10_np([(k >> np.uint64(2)) & np.uint64(0xffffffff), np.zeros_like(k), np.full_like(k, instance), np.zeros_like(k)],
                         [int(seed) & 0xffffffff, (int(seed) >> 32) & 0xffffffff])
    w = np.choose((k & np.uint64(3)).astype(np.int64), c)
    return ((w >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)).astype(np.float32)


def _obs_diff(what, g, o):
    bad = [(a, c, int((g[a][c] != o[a][c]).sum())) for a in range(o.shape[0]) for c in range(o.shape[1])
           if not np.array_equal(g[a][c], o[a][c])]
    return f"{what}: obs differs (agent, channel, #cells): {bad[:8]}"


def run_parity(cfg_kwargs, seeds, steps, p_feed=1 / 3, p_split=1 / 3, boost=None, obs_every=5, replay_len=1 << 16,
               with_obs_in_step=True, ram=False, philox=False, state_every=1, instance_base=0, obs_ref=None, edit=None,
               via="step"):
    """Runs len(seeds) instances on the GPU in one batch and each one through the oracle.
    philox: the GPU draws from its own counter-based Philox stream (AGARCL_RNG_PHILOX, what bench.py runs) and the oracle is
    fed the same stream computed by philox_uniform_np; otherwise both replay the mt19937_64 stream of the seed.
    state_every: the full state is compared every that many steps (rewards and dones every step).
    obs_ref: applied to the oracle's int32 frames before they are compared (int16: np.clip to the int16 range, which is
    exact because every scatter operation is monotone).
    edit(i, state_view): applied to the oracle's and the device's state of instance i after the reset, before the first step.
    via: "step" (Batch.step), "mirror" (Batch.step_mirror; the host mirror is compared with the oracle as well) or "lists"
    (Batch.step_lists; every image of ObsLists.expand and the numpy decoder on a sample are compared with the oracle).
    The returned stats hold the launch counts seen (`launches`, sorted)."""
    oracle_lib().oracle_set_trig_mode(1)
    n = len(seeds)
    if philox:
        from agarcl_b200 import RNG_PHILOX
        cfg = make_cfg(n_instances=n, rng_mode=RNG_PHILOX, ram_obs=ram, instance_base=instance_base, **cfg_kwargs)
        ocfg = make_cfg(n_instances=n, rng_mode=RNG_REPLAY, cap_replay=replay_len, ram_obs=ram, instance_base=instance_base, **cfg_kwargs)
    else:
        cfg = ocfg = make_cfg(n_instances=n, rng_mode=RNG_REPLAY, cap_replay=replay_len, ram_obs=ram, **cfg_kwargs)
    b = Batch(cfg)
    L = b.layout
    Lo = oracle_layout(ocfg)
    if not philox:
        assert bytes(L) == bytes(Lo), "product and oracle layouts differ"
    oras = []
    for i, s in enumerate(seeds):
        o = Oracle(ocfg, Lo)
        if philox:
            o.set_replay(philox_uniform_np(s, instance_base + i, np.arange(replay_len)))
        else:
            o.seed_mt(s, replay_len)
            b.set_replay(i, o.replay)
        oras.append(o)
    b.seed(np.asarray(seeds, dtype=np.uint64))
    b.reset()
    if ocfg.strict_reference:  # the player order the batch's reset made (quirk Q3)
        for k in range(L.P):
            Lo.order[k] = b.layout.order[k]
    for o in oras:
        o.reset()
    if boost:
        for i, o in enumerate(oras):
            for a in range(L.A):
                o.state.cells[a][0]["mass"] = boost
            sv = b.download_state(i)
            for a in range(L.A):
                sv.cells[a][0]["mass"] = boost
            b.upload_state(i, sv)
    if edit:
        for i, o in enumerate(oras):
            edit(i, o.state)
            sv = b.download_state(i)
            edit(i, sv)
            b.upload_state(i, sv)
    for i, o in enumerate(oras):
        d = compare_states(o.state, b.download_state(i))
        assert not d, f"reset mismatch inst {i}: {d[:5]}"
    import torch
    obs_t = b.obs_tensor()
    rew_t = b.rewards_tensor()
    done_t = b.dones_tensor()
    ram_t = b.ram_tensor() if ram else None
    if ram:
        for o in oras:
            o.ram_clear()
    rngs = [np.random.default_rng(s) for s in seeds]
    A = L.A
    launches = set()
    h_rew, h_done = np.zeros(n * A, np.float64), np.zeros(n * A, np.uint8)
    for st in range(steps):
        dxdy = np.zeros((n, A, 2), np.float32)
        act = np.zeros((n, A), np.int32)
        for i in range(n):
            dxdy[i], act[i] = random_actions(rngs[i], A, p_feed, p_split)
        if via == "step":
            b.set_actions(dxdy, act)
            b.step()
        elif via == "mirror":
            h_obs = b.step_mirror(dxdy, act, h_rew, h_done).reshape(n, A, *b.obs_shape[1:])
        elif via == "lists":
            lists = b.step_lists(dxdy, act, h_rew, h_done)
        else:
            raise ValueError(f"via={via!r}")
        launches.add(b.launches_per_step())
        torch.cuda.synchronize()
        g_rew = rew_t.cpu().numpy().reshape(n, A)
        g_done = done_t.cpu().numpy().reshape(n, A)
        if via != "step":  # what the host copy of the step handed out
            assert np.array_equal(h_rew.reshape(n, A), g_rew) and np.array_equal(h_done.reshape(n, A), g_done), f"step {st}: {via} rewards / dones"
        want_obs = (st % obs_every == 0)
        g_obs = obs_t.cpu().numpy().reshape(n, A, *b.obs_shape[1:]) if want_obs else None
        g_ram = ram_t.cpu().numpy() if ram else None
        for i, o in enumerate(oras):
            o.set_actions(dxdy[i], act[i])
            o_rew, o_done, o_obs = (o.step_with_ram(with_obs=want_obs and with_obs_in_step) if ram
                                    else o.step(with_obs=want_obs and with_obs_in_step))
            if st % state_every == 0 or st == steps - 1:
                gs = b.download_state(i)
                d = compare_states(o.state, gs)
                assert not d, f"step {st} inst {i} (seed {seeds[i]}): {d[:6]} flags gpu={gs.flag_names()} oracle={o.state.flag_names()}"
                assert int(gs.hdr["flags"]) == int(o.state.hdr["flags"]), (st, i, gs.flag_names(), o.state.flag_names())
                assert int(gs.hdr["rng_cursor"]) == int(o.state.hdr["rng_cursor"]), (st, i)
            assert np.array_equal(g_rew[i], o_rew), f"step {st} inst {i}: rewards {g_rew[i]} vs {o_rew}"
            assert np.array_equal(g_done[i], o_done), f"step {st} inst {i}: dones {g_done[i]} vs {o_done}"
            if ram:
                same = (g_ram[i].view(np.uint32) == o.ram.view(np.uint32)) | (np.isnan(g_ram[i]) & np.isnan(o.ram))
                if not same.all():
                    bad = np.argwhere(~same)[:8].tolist()
                    raise AssertionError(f"step {st} inst {i}: ram records differ at (player, slot) {bad}: "
                                         f"{[(float(g_ram[i][p, k]), float(o.ram[p, k])) for p, k in bad]}")
            if want_obs:
                if o_obs is None:
                    o_obs = np.stack([o.obs(a) for a in range(A)])
                if obs_ref is not None:
                    o_obs = obs_ref(o_obs)
                if not np.array_equal(g_obs[i], o_obs):
                    bad = [(a, c, int((g_obs[i][a][c] != o_obs[a][c]).sum())) for a in range(A) for c in range(o_obs.shape[1])
                           if not np.array_equal(g_obs[i][a][c], o_obs[a][c])]
                    raise AssertionError(f"step {st} inst {i}: obs differs (agent, channel, #cells): {bad[:8]}")
                if via == "mirror" and not np.array_equal(h_obs[i], o_obs):
                    raise AssertionError(_obs_diff(f"step {st} inst {i}: host mirror", h_obs[i], o_obs))
                if via == "lists":
                    ex = np.stack([lists.expand(i * A + a) for a in range(A)])
                    if not np.array_equal(ex, o_obs):
                        raise AssertionError(_obs_diff(f"step {st} inst {i}: lists (C decoder)", ex, o_obs))
                    dec = lists.decode(i * A + st % A)  # (slow: one image per instance and step; None: it took the dense copy)
                    assert dec is None or np.array_equal(dec, o_obs[st % A]), f"step {st} inst {i}: lists (numpy decoder)"
    stats = dict(cells_eaten=sum(int(o.state.players["cells_eaten"].sum()) for o in oras),
                 viruses_eaten=sum(int(o.state.players["viruses_eaten"].sum()) for o in oras),
                 food_eaten=sum(int(o.state.players["food_eaten"].sum()) for o in oras),
                 max_cells=max(int(o.state.players["n_cells"].max()) for o in oras),
                 foods=sum(int(o.state.hdr["n_foods"]) for o in oras),
                 flags=sorted({f for o in oras for f in o.state.flag_names()}),
                 launches=sorted(launches))
    b.close()
    return stats
