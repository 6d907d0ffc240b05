"""Mixed-task batches (cfg.task_modes, include/agarcl_b200.h): an instance of mode m in a batch of all ten mini-games steps bit for
bit like the same instance of a batch of mode m alone, and like the oracle of its mode; a new task starts at the instance's next
reset and not before; bad tasks are rejected per instance on the device; nothing makes the host wait; snapshots carry the task."""
import numpy as np
import pytest

from agarcl_b200 import RNG_MT19937, RNG_REPLAY, make_cfg
from agarcl_b200._abi import StateView, compare_states, task_bits
from gpu_parity_lib import assert_no_host_wait, i32

MODES = list(range(1, 11))
# the ten AgarCL mini-games (bench/tasks_configs): arena 350, 500 pellets, no viruses, one bot in modes 7..10
MINI = dict(arena_size=350, num_pellets=500, num_viruses=0, num_bots=0, grid_size=64)
SEEDS_BASE, BASE = 500, 300


def mode_of(i):
    return MODES[i % 10]


def project(sv, L):
    """the state of `sv` in layout L (fewer players or another pellet capacity): the fields a game of L's players holds"""
    out = StateView(L)
    out.blob[L.off_hdr:L.off_hdr + 64] = sv.blob[sv.layout.off_hdr:sv.layout.off_hdr + 64]
    out.players[:] = sv.players[:L.P]
    out.cells[:] = sv.cells[:L.P]
    nv, nf, npl = min(L.cap_viruses, sv.layout.cap_viruses), min(L.cap_foods, sv.layout.cap_foods), min(L.cap_pellets, sv.layout.cap_pellets)
    out.viruses[:nv] = sv.viruses[:nv]
    out.foods[:nf] = sv.foods[:nf]
    out.pellets[:npl] = sv.pellets[:npl]
    return out


HDR = ("rng_cursor", "next_cell_id", "flags", "seed_lo", "seed_hi", "respawned_lo", "respawned_hi")


def assert_same_game(mixed_sv, alone_sv, what, hdr=HDR):
    """field by field: header, players < P_m and their cells, viruses, foods, the first n_pellets pellets"""
    p = project(mixed_sv, alone_sv.layout)
    d = compare_states(p, alone_sv)
    assert not d, f"{what}: {d[:6]}"
    for f in hdr:
        assert int(p.hdr[f]) == int(alone_sv.hdr[f]), (what, f)


def make_mixed(N, modes=None, limits=None, **kw):
    """a batch of the ten mini-games, instance i on modes[i] (default 1 + i % 10) from its first reset on"""
    from agarcl_b200.batch import Batch
    b = Batch(make_cfg(n_instances=N, mode_number=1, task_modes=task_bits(MODES), instance_base=BASE, **dict(MINI, **kw)))
    b.seed(np.arange(N, dtype=np.uint64) + SEEDS_BASE)
    res = b.set_tasks(i32(modes if modes is not None else [mode_of(i) for i in range(N)]), i32(limits) if limits is not None else None)
    assert (res.cpu().numpy() == 1).all()
    return b


def make_alone(N, m, **kw):
    from agarcl_b200.batch import Batch
    b = Batch(make_cfg(n_instances=N, mode_number=m, instance_base=BASE, **dict(MINI, **kw)))
    b.seed(np.arange(N, dtype=np.uint64) + SEEDS_BASE)
    return b


def _check_step(mixed, alone, N, what, state=True):
    """obs, rewards, dones, ram records (players < P_m) and -- with `state` -- the game of every instance against its twin"""
    import torch
    torch.cuda.synchronize()
    A = mixed.A
    mo, mr, md = mixed.obs_tensor().cpu().numpy(), mixed.rewards_tensor().cpu().numpy(), mixed.dones_tensor().cpu().numpy()
    al = {m: (b.obs_tensor().cpu().numpy(), b.rewards_tensor().cpu().numpy(), b.dones_tensor().cpu().numpy()) for m, b in alone.items()}
    ram = mixed.ram_tensor().cpu().numpy() if mixed.cfg.ram_obs else None
    for i in range(N):
        m = mode_of(i)
        s = slice(i * A, (i + 1) * A)
        assert np.array_equal(mo[s], al[m][0][s]), f"{what}: obs of instance {i} (mode {m})"
        assert np.array_equal(mr[s], al[m][1][s]) and np.array_equal(md[s], al[m][2][s]), f"{what}: reward / done of {i} (mode {m})"
        if ram is not None:
            ra = alone[m].ram_tensor().cpu().numpy()
            assert np.array_equal(ram[i, :alone[m].layout.P], ra[i]), f"{what}: ram records of {i}"
        if state:
            assert_same_game(mixed.download_state(i), alone[m].download_state(i), f"{what}: instance {i} (mode {m})")


def _actions(rng, n):
    return rng.uniform(-1, 1, size=(n, 2)).astype(np.float32), rng.integers(0, 3, size=n).astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["step", "step_autoreset", "mt19937", "step_lists"])
def test_mixed_batch_equals_ten_single_mode_batches(path):
    """N instances, instance i on mode 1 + i % 10, against ten batches of one mode each with the same N, seeds, instance_base and
    actions: instance i of the mixed batch is instance i of the batch of its mode, bit for bit"""
    N = 20
    kw = dict(ram_obs=1) if path == "step" else {}
    if path == "mt19937":
        kw = dict(rng_mode=RNG_MT19937)
    steps = {"step": 300, "step_autoreset": 200, "mt19937": 100, "step_lists": 40}[path]
    limit = {m: (40, 60, 80)[m % 3] for m in MODES}  # short episodes: truncations (and bot kills) reset within the run
    mixed = make_mixed(N, limits=[limit[mode_of(i)] for i in range(N)] if path == "step_autoreset" else None, **kw)
    alone = {m: make_alone(N, m, **kw) for m in MODES}
    for b in [mixed] + list(alone.values()):
        b.reset()
        if path == "step_autoreset":
            b.set_autoreset(limit[b.cfg.mode_number] if b is not mixed else 1000)
    _check_step(mixed, alone, N, "after reset")
    rng = np.random.default_rng(3)
    resets = 0
    for t in range(steps):
        acts = _actions(rng, N * mixed.A)
        if path == "step_lists":
            lists = {m: b.step_lists(*acts) for m, b in alone.items()}
            ml = mixed.step_lists(*acts)
            for i in range(N):
                assert np.array_equal(ml.expand(i), lists[mode_of(i)].expand(i)), f"step {t}: lists of instance {i}"
                assert ml.rewards_dones()[0][i] == lists[mode_of(i)].rewards_dones()[0][i]
        else:
            for b in [mixed] + list(alone.values()):
                b.set_actions(*acts)
                b.step_autoreset() if path == "step_autoreset" else b.step()
        if path == "step_autoreset":
            me = {k: v.cpu().numpy() for k, v in mixed.episode().items()}
            resets += int(me["reset_mask"].sum())
            for i in range(N):
                ae = alone[mode_of(i)].episode()
                for k in ("done", "reset_mask", "steps", "episode_length", "episode_return"):
                    if k in ("episode_length", "episode_return") and not me["reset_mask"][i]:
                        continue
                    assert me[k][i] == ae[k].cpu().numpy()[i], f"step {t}: episode {k} of {i}"
        _check_step(mixed, alone, N, f"{path} step {t}", state=(t % 20 == 19 or t == steps - 1))
    if path == "step_autoreset":
        assert resets >= N, "the per-instance limits did not end episodes"
        assert (mixed.tasks()["mode"].cpu().numpy() == [mode_of(i) for i in range(N)]).all()
    assert mixed.flags()[0] == 0
    for b in [mixed] + list(alone.values()):
        b.close()


def _oracle_for(mode, i, seed, replay_len=1 << 16):
    from _helpers import Oracle, oracle_layout
    from gpu_parity_lib import philox_uniform_np
    ocfg = make_cfg(n_instances=1, mode_number=mode, rng_mode=RNG_REPLAY, cap_replay=replay_len, instance_base=BASE + i, **MINI)
    o = Oracle(ocfg, oracle_layout(ocfg))
    o.set_replay(philox_uniform_np(seed, BASE + i, np.arange(replay_len)))
    o.state.hdr["seed_lo"], o.state.hdr["seed_hi"] = seed & 0xFFFFFFFF, seed >> 32  # (kept by the oracle's reset)
    return o


def _step_against_oracles(b, oras, K, rng, what):
    import torch
    A = b.A
    for st in range(K):
        dxdy, act = _actions(rng, b.N * A)
        b.set_actions(dxdy, act)
        b.step()
        torch.cuda.synchronize()
        g_rew = b.rewards_tensor().cpu().numpy().reshape(b.N, A)
        g_done = b.dones_tensor().cpu().numpy().reshape(b.N, A)
        g_obs = b.obs_tensor().cpu().numpy().reshape(b.N, A, *b.obs_shape[1:])
        for i, o in oras.items():
            o.set_actions(dxdy[i * A:(i + 1) * A], act[i * A:(i + 1) * A])
            o_rew, o_done, o_obs = o.step(with_obs=True)
            gs = project(b.download_state(i), o.L)
            d = compare_states(o.state, gs)
            assert not d, f"{what} step {st} inst {i}: {d[:6]}"
            assert int(gs.hdr["rng_cursor"]) == int(o.state.hdr["rng_cursor"]) and int(gs.hdr["flags"]) == int(o.state.hdr["flags"])
            assert np.array_equal(g_rew[i], o_rew) and np.array_equal(g_done[i], o_done), (what, st, i)
            assert np.array_equal(g_obs[i], o_obs), f"{what} step {st} inst {i}: obs"


@pytest.mark.gpu
def test_mixed_instances_against_the_oracle_of_their_mode():
    """instance 0 (mode 1: its bot slot is absent) and instance 6 (mode 7: one bot) of a mixed batch, each against the oracle of
    its own mode reset on the same Philox stream (seed, global index)"""
    from _helpers import oracle_lib
    oracle_lib().oracle_set_trig_mode(1)
    N = 10
    b = make_mixed(N)
    b.reset()
    assert b.layout.P == 2
    oras = {}
    for i in (0, 6):
        o = _oracle_for(mode_of(i), i, SEEDS_BASE + i)
        o.reset()
        assert_same_game(b.download_state(i), o.state, f"reset of instance {i}", HDR[:5])
        oras[i] = o
    st = b.download_state(0)
    assert int(st.players["n_cells"][1]) == 0 and int(st.hdr["next_cell_id"]) == 2  # the absent player, cell ids of one player
    _step_against_oracles(b, oras, 120, np.random.default_rng(4), "mixed")
    b.close()


@pytest.mark.gpu
def test_a_new_task_starts_at_the_next_reset():
    """set_tasks changes nothing until the instance's next reset (a twin without the call stays bit-identical); from that reset on
    the instance plays the new mode: the oracle of that mode fed the instance's stream from its cursor"""
    import torch
    from _helpers import oracle_lib
    oracle_lib().oracle_set_trig_mode(1)
    N = 10
    a, twin = make_mixed(N), make_mixed(N)
    rng = np.random.default_rng(6)
    for b in (a, twin):
        b.reset()
    switch = {0: 8, 3: 2, 7: 5}  # instance: new mode
    new = [switch.get(i, -1) for i in range(N)]
    res = a.set_tasks(i32(new), i32([25 if i in switch else -1 for i in range(N)]))
    assert res.cpu().numpy().tolist() == [1] * N  # (a limit of -1 is a value too: every entry was set)
    t = a.tasks()
    assert t["mode"].cpu().numpy().tolist() == [mode_of(i) for i in range(N)]
    assert t["next_mode"].cpu().numpy().tolist() == [switch.get(i, mode_of(i)) for i in range(N)]
    for _ in range(15):
        acts = _actions(rng, N)
        for b in (a, twin):
            b.set_actions(*acts)
            b.step()
    torch.cuda.synchronize()
    for i in range(N):
        assert np.array_equal(a.download_state(i).blob, twin.download_state(i).blob), i
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
    mask[list(switch)] = 1
    a.reset_device(mask)
    torch.cuda.synchronize()
    assert t["mode"].cpu().numpy().tolist() == [switch.get(i, mode_of(i)) for i in range(N)]
    assert t["max_steps"].cpu().numpy().tolist() == [25 if i in switch else -1 for i in range(N)]
    oras = {}
    for i, m in switch.items():
        o = _oracle_for(m, i, SEEDS_BASE + i)
        # the oracle's reset of mode m from the cursor the instance stood at (its stream goes on: Engine::reset does not reseed)
        o.state.hdr["rng_cursor"] = twin.download_state(i).hdr["rng_cursor"]
        o.reset_keep_stream()
        assert_same_game(a.download_state(i), o.state, f"reset of instance {i} into mode {m}", HDR[:5])
        oras[i] = o
    for i in range(N):
        if i not in switch:
            assert np.array_equal(a.download_state(i).blob, twin.download_state(i).blob), i
    _step_against_oracles(a, oras, 60, np.random.default_rng(7), "switched")
    a.close()
    twin.close()


@pytest.mark.gpu
def test_vector_env_tasks_and_episode_lengths():
    """BatchedAgarioEnv(tasks=...): info["task"] is the current mode (after an auto-reset the new episode's), and a truncated
    episode ends on its instance's own limit, as a batch-wide limit of the same value ends it (limit + 1 steps: the limit is
    checked before the step is counted, like gym_agario's AgarioEnv.step)"""
    import torch
    from agarcl_b200.gym_env import BatchedAgarioEnv
    N = 12
    env = BatchedAgarioEnv(N, tasks=[1, 2, 4, 6], number_steps=500, **MINI)
    env.seed(3)
    modes = [(1, 2, 4, 6)[i % 4] for i in range(N)]
    lim = [(30, 45, 0, -1)[i % 4] if i < 8 else 20 for i in range(N)]
    assert (env.set_tasks(i32(modes), i32(lim)).cpu().numpy() == 1).all()
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(0)
    seen_len = {i: set() for i in range(N)}
    for t in range(100):
        if t == 50:  # instances 8.. switch to mode 2 at their next truncation
            assert (env.set_tasks(i32([-1] * 8 + [2] * (N - 8))).cpu().numpy() == [0] * 8 + [1] * (N - 8)).all()
        _, _, done, _, info = env.step((torch.rand((N, 2), device="cuda", generator=g) * 2 - 1), torch.zeros(N, dtype=torch.int32, device="cuda"))
        m = info["reset_mask"].cpu().numpy()
        L = info["episode_length"].cpu().numpy()
        task = info["task"].cpu().numpy()
        for i in np.flatnonzero(m):
            seen_len[i].add(int(L[i]))
        want_task = [modes[i] if (i < 8 or t < 62) else 2 for i in range(N)]
        for i in range(N):  # (instances 8.. truncate at steps 20, 41, 62, 83: the first reset after the call is at 62)
            assert task[i] == want_task[i], (t, i, task[i])
    for i in range(N):
        want = {lim[i] + 1} if lim[i] > 0 else set()  # 0: no limit; -1: number_steps = 500, beyond the run
        assert seen_len[i] == want, (i, seen_len[i])
    env.close()


@pytest.mark.gpu
def test_rejections_and_refusals():
    import torch
    from agarcl_b200._lib import AgarclError
    from agarcl_b200.batch import Batch
    N = 6
    b = make_mixed(N, modes=[1] * N)
    b.reset()
    before = {k: v.clone() for k, v in b.tasks().items()}
    res = b.set_tasks(i32([11, 0, -1, 3, -1, -2]), i32([10, 10, -2, -1, -1, 5]))
    torch.cuda.synchronize()
    # mode 11 / mode 0 (not in the set) / limit -2 / fine / limit only / mode -2
    assert res.cpu().numpy().tolist() == [2, 2, 2, 1, 1, 2]
    t = b.tasks()
    assert t["next_mode"].cpu().numpy().tolist() == [1, 1, 1, 3, 1, 1]
    assert t["next_max_steps"].cpu().numpy().tolist() == [-1, -1, -1, -1, -1, -1]
    assert torch.equal(t["mode"], before["mode"]) and torch.equal(t["max_steps"], before["max_steps"])
    assert b.set_tasks(i32([-1] * N)).cpu().numpy().tolist() == [0] * N
    with pytest.raises(AgarclError, match="mode"):
        b.set_tasks(i32([1] * (N - 1)))
    b.close()
    plain = Batch(make_cfg(n_instances=2, mode_number=1, **MINI))
    with pytest.raises(AgarclError, match="without task_modes"):
        plain.set_tasks(i32([1, 1]))
    with pytest.raises(AgarclError, match="without task_modes"):
        plain.tasks()
    plain.close()
    for kw, msg in [(dict(strict_reference=1), "strict_reference"), (dict(mode_number=0), "mode 0"),
                    (dict(task_modes=task_bits([2, 3])), "must contain mode_number 1")]:
        cfg = dict(MINI, n_instances=2, mode_number=1, task_modes=task_bits(MODES))
        cfg.update(kw)
        if kw.get("mode_number") == 0:
            cfg["task_modes"] = task_bits([0] + MODES)
        with pytest.raises(AgarclError, match=msg):
            Batch(make_cfg(**cfg))


@pytest.mark.gpu
def test_set_tasks_and_step_autoreset_do_not_wait_for_the_device():
    import torch
    N = 64
    b = make_mixed(N)
    b.reset()
    b.set_autoreset(50)
    modes = i32([mode_of(i + 1) for i in range(N)])
    s = torch.cuda.Stream()
    for _ in range(2):  # every kernel on the path is loaded before the timed calls
        b.set_tasks(modes, stream=s.cuda_stream)
        b.step_autoreset(stream=s.cuda_stream)

    def calls():
        b.set_tasks(modes, stream=s.cuda_stream)
        b.step_autoreset(stream=s.cuda_stream)

    assert_no_host_wait(calls, s)
    b.close()


@pytest.mark.gpu
def test_snapshots_carry_the_task(tmp_path):
    """a mode-8 state restored into a mode-2 instance at the same global index continues bit for bit like its source and reports
    mode 8; pools of batches with and without tasks reject each other's slots; the JSON snapshot keeps the mode"""
    import torch
    from agarcl_b200._lib import AgarclError
    from agarcl_b200.batch import Batch
    N, j = 10, 7  # instance 7 plays mode 8
    src = make_mixed(N)
    dst = make_mixed(N, modes=[2] * N)
    rng = np.random.default_rng(8)
    for b in (src, dst):
        b.reset()
    for _ in range(20):
        acts = _actions(rng, N)
        for b in (src, dst):
            b.set_actions(*acts)
            b.step()
    pool = src.snapshot_pool(1)
    src.save_states(pool, i32([j]))
    res = dst.restore_states(pool, i32([0 if i == j else -1 for i in range(N)]))
    torch.cuda.synchronize()
    assert res.cpu().numpy().tolist() == [1 if i == j else 0 for i in range(N)]
    t = dst.tasks()
    assert int(t["mode"][j]) == 8 and int(t["next_mode"][j]) == 2  # the pending task is the destination's own
    hdr = pool[0, :64].cpu().numpy().view(np.int32)
    assert hdr[7] == 8 and hdr[8] == -1  # agarcl_snapshot_hdr.task_mode, task_max_steps
    for st in range(40):
        acts = _actions(rng, N)
        for b in (src, dst):
            b.set_actions(*acts)
            b.step()
        torch.cuda.synchronize()
        assert np.array_equal(src.download_state(j).blob, dst.download_state(j).blob), st
        assert np.array_equal(src.obs_tensor()[j].cpu().numpy(), dst.obs_tensor()[j].cpu().numpy()), st
    # slots of a batch without tasks and of a mixed batch of the same layout (modes 7 and 8: P = 2, 500 pellets) reject each other
    mixed78 = Batch(make_cfg(n_instances=2, mode_number=7, task_modes=task_bits([7, 8]), **MINI))
    plain7 = Batch(make_cfg(n_instances=2, mode_number=7, **MINI))
    assert mixed78.slot_bytes == plain7.slot_bytes
    for b in (mixed78, plain7):
        b.reset()
    for a, b in ((mixed78, plain7), (plain7, mixed78)):
        p = a.snapshot_pool(1)
        a.save_states(p, i32([0]))
        assert b.restore_states(p, i32([0, -1])).cpu().numpy().tolist() == [2, 0]
        assert a.restore_states(p, i32([-1, 0])).cpu().numpy().tolist() == [0, 1]
    # JSON: the instance's current mode travels as mode_number and comes back as the loading instance's current task
    path = tmp_path / "mode8.json"
    src.save_env_state(j, path)
    import json
    with open(path) as f:
        js = json.load(f)
    assert js["mode_number"] == 8 and len(js["players"]) == 2
    dst.load_env_state(1, path, lossless=True)
    assert int(dst.tasks()["mode"][1]) == 8
    assert_same_game(dst.download_state(1), src.download_state(j), "JSON load")
    path2 = tmp_path / "mode2.json"
    dst.save_env_state(2, path2)
    with open(path2) as f:
        js = json.load(f)
    assert js["mode_number"] == 2 and len(js["players"]) == 1
    src.load_env_state(6, path2, lossless=True)  # instance 6 (mode 7, a live bot) takes the one-player mode-2 game
    st = src.download_state(6)
    assert int(src.tasks()["mode"][6]) == 2 and int(st.players["n_cells"][1]) == 0
    with pytest.raises(AgarclError, match="not in the batch's task_modes"):
        mixed78.load_env_state(0, path2)
    for b in (src, dst, mixed78, plain7):
        b.close()
