"""The pixel observation (cfg.pixel_obs, k_draw_views in draw_kernel.cu): every agent's picture after every step, reset and
restore is byte-exact against oracle_draw's agent view on the downloaded blob with the respawned players' cells removed; the
game is the same as with the grid observation; auto-reset with final pictures, masked resets and restores rewrite exactly
their instances; pools move between pixel and grid batches; the crafted maximal state; no host wait; the refusals and the
Python layers."""
import ctypes as C

import numpy as np
import pytest

from _helpers import AGENT, oracle_draw
from agarcl_b200 import make_cfg
from agarcl_b200._abi import StateView
from gpu_parity_lib import CASES, assert_no_host_wait, device_record, i32

# name: (make_cfg keywords, p_feed, p_split, boost); CASES entries plus the games these tests need beyond them
PIXEL_CASES = dict(CASES)
PIXEL_CASES.update({
    # small and crowded: bots eat the agents, and mode 0 respawns them
    "mode0_respawns": (dict(num_agents=2, num_bots=10, arena_size=150, num_pellets=200, num_viruses=2), 0.2, 0.2, None),
    # agents of mass 1000: a 300-unit window in a 350-unit arena holds nearly everything
    "mode5": (dict(mode_number=5, num_bots=0), 1 / 3, 1 / 3, None),
    "mode6": (dict(mode_number=6, num_bots=0), 1 / 3, 1 / 3, None),
})


def pixel_batch(name, S, N=4, seed=5, **more):
    from agarcl_b200.batch import Batch
    kw, p_feed, p_split, boost = PIXEL_CASES[name]
    b = Batch(make_cfg(n_instances=N, pixel_obs=S, **kw, **more))
    b.seed(seed)
    if b.cfg.task_modes:
        b.set_tasks(i32([1, 7, 8, 10][:N] + [1] * max(0, N - 4)))
    b.reset()
    return b, np.random.default_rng(seed), p_feed, p_split, boost


def boost_agents(b, boost):
    """the agents' first cell gets mass `boost`; the pictures are drawn again by a restore of the boosted states into themselves"""
    import torch
    for i in range(b.N):
        sv = b.download_state(i)
        for a in range(b.A):
            sv.cells[a][0]["mass"] = boost
        b.upload_state(i, sv)
    redraw(b)
    torch.cuda.synchronize()


def redraw(b):
    pool = b.snapshot_pool(b.N)
    b.save_states(pool, i32(range(b.N)))
    assert b.restore_states(pool, i32(range(b.N))).cpu().numpy().tolist() == [1] * b.N


def expected(b, blob, agent, pre_respawn=True):
    """the spec: oracle_draw's agent view with the players of hdr.respawned_lo / _hi drawn without cells"""
    blob = blob.copy()
    if pre_respawn:
        sv = StateView(b.layout, blob)
        m = int(sv.hdr["respawned_lo"]) | int(sv.hdr["respawned_hi"]) << 32
        for p in range(b.layout.P):
            if (m >> p) & 1:
                sv.players["n_cells"][p] = 0
    return oracle_draw(b.cfg, b.layout, blob, AGENT, agent, b.cfg.pixel_obs)


def check(b, pics=None, instances=None, pre_respawn=True, what=""):
    import torch
    torch.cuda.synchronize()
    pics = (b.pixels() if pics is None else pics).cpu().numpy()
    for i in range(b.N) if instances is None else instances:
        blob = b.download_state(i).blob
        for a in range(b.A):
            exp = expected(b, blob, a, pre_respawn)
            got = pics[i * b.A + a]
            if not np.array_equal(got, exp):
                bad = np.argwhere(np.any(got != exp, axis=-1))
                raise AssertionError(f"{what} instance {i} agent {a}: {len(bad)} pixels differ, first {bad[:4].tolist()}: "
                                     f"{got[tuple(bad[0])]} vs {exp[tuple(bad[0])]}")


def respawn_mask(b, i):
    sv = b.download_state(i)
    return int(sv.hdr["respawned_lo"]) | int(sv.hdr["respawned_hi"]) << 32


def random_step(b, rng, p_feed, p_split):
    from _helpers import random_actions
    b.set_actions(*random_actions(rng, b.N * b.A, p_feed, p_split))
    b.step()


RUNS = [("c2", 128), ("c2", 48), ("c4_four_agents", 64), ("c4_four_agents", 256), ("mode0_respawns", 16),
        ("mode0_respawns", 128), ("mode1", 48), ("mode1", 64), ("mode5", 128), ("mode5", 256), ("mode6", 64), ("mode6", 16),
        ("mixed_tasks", 128), ("mixed_tasks", 48)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,S", RUNS)
def test_pictures_match_oracle_every_step(name, S):
    b, rng, p_feed, p_split, boost = pixel_batch(name, S)
    check(b, what="after the reset")
    if boost:
        boost_agents(b, boost)
        check(b, what="boosted")
    respawns = 0
    for t in range(200):
        random_step(b, rng, p_feed, p_split)
        check(b, what=f"step {t}")
        respawns += sum(bin(respawn_mask(b, i)).count("1") for i in range(b.N)) if name == "mode0_respawns" else 0
    if name == "mode0_respawns":
        assert respawns > 0, "no player was respawned: the case does not test pre_respawn"
    if name == "c4_four_agents":
        assert max(int(b.download_state(i).players["n_cells"][:b.A].max()) for i in range(b.N)) > 1
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("ram", [0, 1])
def test_game_unchanged_by_pixels(ram):
    """a pixel batch and a grid batch of one configuration, seeds and actions hold the same states, rewards, dones (and ram
    records) every step"""
    from _helpers import random_actions
    from agarcl_b200.batch import Batch
    kw = dict(n_instances=6, num_agents=2, ram_obs=ram, num_bots=8, arena_size=300, num_pellets=300, num_viruses=4)
    pix, grid = Batch(make_cfg(pixel_obs=64, **kw)), Batch(make_cfg(**kw))
    for b in (pix, grid):
        b.seed(11)
        b.reset()
    rng = np.random.default_rng(2)
    for t in range(150):
        acts = random_actions(rng, 12, 0.3, 0.3)
        for b in (pix, grid):
            b.set_actions(*acts)
            b.step()
        p, g = device_record(pix), device_record(grid)
        for k in g:
            if k != "obs":
                assert np.array_equal(p[k], g[k]), f"step {t}: {k}"
        assert not p["obs"].any(), "a pixel batch renders no grid frame"
    check(pix, what="last step")


@pytest.mark.gpu
def test_autoreset_final_pictures():
    """final pictures are the oracle's pictures of the finished state (a twin pixel batch stepped with plain step()); the
    observation after the reset is the new episode's first picture; instances not reset keep their picture bit for bit"""
    import torch
    from _helpers import random_actions
    b, rng, pf, ps, _ = pixel_batch("mode9_deaths_and_limit", 64, N=8)
    twin, _, _, _, _ = pixel_batch("mode9_deaths_and_limit", 64, N=8)
    b.set_autoreset(25, keep_final_obs=True)
    finals = 0
    for t in range(120):
        acts = random_actions(rng, b.N * b.A, pf, ps)
        for x in (b, twin):
            x.set_actions(*acts)
        b.step_autoreset()
        twin.step()
        torch.cuda.synchronize()
        rm = b.episode()["reset_mask"].cpu().numpy()
        fin, tw = b.final_pixels().cpu().numpy(), twin.pixels().cpu().numpy()
        for i in np.flatnonzero(rm):
            finals += 1
            for a in range(b.A):
                j = i * b.A + a
                assert np.array_equal(fin[j], tw[j]), f"step {t} instance {i}: final picture"
            check(twin, twin.pixels(), instances=[i], what=f"step {t} finishing")
        if rm.any():
            twin.reset(rm)
        cur, tw = b.pixels().cpu().numpy(), twin.pixels().cpu().numpy()
        assert np.array_equal(cur, tw), f"step {t}: pictures differ from the twin's"
        if t % 10 == 0 or rm.any():
            check(b, what=f"step {t} after auto-reset")
    assert finals > 2
    assert_no_host_wait(lambda: [b.step_autoreset() for _ in range(3)], torch.cuda.current_stream())


@pytest.mark.gpu
def test_masked_resets_and_restores_rewrite_only_their_instances():
    import torch
    b, rng, pf, ps, _ = pixel_batch("c2", 48, N=6)
    for _ in range(30):
        random_step(b, rng, pf, ps)
    for how in ("host", "device"):
        before = b.pixels().clone()
        mask = np.array([1, 0, 0, 1, 0, 1] if how == "host" else [0, 1, 1, 0, 0, 0], np.uint8)
        if how == "host":
            b.reset(mask)
        else:
            b.reset_device(torch.as_tensor(mask, device="cuda"))
        after = b.pixels().clone()
        torch.cuda.synchronize()
        for i in range(b.N):
            sl = slice(i * b.A, (i + 1) * b.A)
            if not mask[i]:
                assert torch.equal(before[sl], after[sl]), f"{how} reset touched instance {i}"
        check(b, instances=list(np.flatnonzero(mask)), what=f"{how} reset")
        for _ in range(7):
            random_step(b, rng, pf, ps)
    # restore: a picture comes back as the source showed it at the save
    pool = b.snapshot_pool(2)
    b.save_states(pool, i32([1, 4]))
    saved = b.pixels().clone()
    for _ in range(9):
        random_step(b, rng, pf, ps)
    before = b.pixels().clone()
    res = b.restore_states(pool, i32([-1, -1, 0, 1, -1, 0]))
    torch.cuda.synchronize()
    assert res.cpu().numpy().tolist() == [0, 0, 1, 1, 0, 1]
    after = b.pixels()
    for dst, src in ((2, 1), (3, 4), (5, 1)):
        assert torch.equal(after[dst * b.A:(dst + 1) * b.A], saved[src * b.A:(src + 1) * b.A]), (dst, src)
    for i in (0, 1, 4):
        assert torch.equal(after[i * b.A:(i + 1) * b.A], before[i * b.A:(i + 1) * b.A]), i
    check(b, what="after the restore")


@pytest.mark.gpu
def test_pools_move_between_pixel_and_grid_batches():
    """slot bytes and fingerprint do not depend on pixel_obs: a grid pool restores into a pixel batch and the other way round"""
    import torch
    from _helpers import random_actions
    from agarcl_b200.batch import Batch
    kw = dict(n_instances=4, num_bots=6, arena_size=300, num_pellets=300, num_viruses=4)
    pix, grid = Batch(make_cfg(pixel_obs=32, **kw)), Batch(make_cfg(**kw))
    assert pix.slot_bytes == grid.slot_bytes
    rng = np.random.default_rng(4)
    for b in (pix, grid):
        b.seed(8)
        b.reset()
    for _ in range(20):
        acts = random_actions(rng, 4, 0.3, 0.3)
        for b in (pix, grid):
            b.set_actions(*acts)
            b.step()
    pools = {}
    for name, b in (("pix", pix), ("grid", grid)):
        pools[name] = b.snapshot_pool(4)
        b.save_states(pools[name], i32([3, 2, 1, 0]))
    torch.cuda.synchronize()
    assert torch.equal(pools["pix"][:, 8:16], pools["grid"][:, 8:16]), "fingerprints differ"
    assert torch.equal(pools["pix"], pools["grid"]), "the saved slots differ"
    for _ in range(5):
        acts = random_actions(rng, 4, 0.3, 0.3)
        for b in (pix, grid):
            b.set_actions(*acts)
            b.step()
    assert pix.restore_states(pools["grid"], i32([0, 1, 2, 3])).cpu().numpy().tolist() == [1] * 4
    assert grid.restore_states(pools["pix"], i32([0, 1, 2, 3])).cpu().numpy().tolist() == [1] * 4
    p, g = device_record(pix), device_record(grid)
    assert np.array_equal(p["blobs"], g["blobs"])
    check(pix, what="grid pool restored into a pixel batch")


@pytest.mark.gpu
def test_crafted_maximal_state_with_and_without_respawned_players():
    """64 players x 32 cells and full pellet, virus and food capacities (more than one pass of both culled lists); half the
    players, agent 1 among them, marked as respawned: draw() shows them (pre_respawn 0), the observation does not (1)"""
    import torch
    from agarcl_b200.batch import Batch
    b = Batch(make_cfg(n_instances=2, num_agents=4, num_bots=60, num_viruses=60, num_pellets=1500, arena_size=600, pixel_obs=128))
    b.seed(1)
    b.reset()
    L = b.layout
    assert L.P == 64
    rng = np.random.default_rng(3)
    sv = b.download_state(0)
    W = 600
    sv.hdr["n_pellets"], sv.hdr["n_viruses"], sv.hdr["n_foods"] = L.cap_pellets, L.cap_viruses, L.cap_foods
    sv.pellets["x"], sv.pellets["y"] = rng.uniform(0, W, L.cap_pellets), rng.uniform(0, W, L.cap_pellets)
    sv.foods["x"], sv.foods["y"] = rng.uniform(0, W, L.cap_foods), rng.uniform(0, W, L.cap_foods)
    sv.viruses["x"], sv.viruses["y"] = rng.uniform(0, W, L.cap_viruses), rng.uniform(0, W, L.cap_viruses)
    sv.viruses["mass"] = rng.choice([100, 150, 200], L.cap_viruses)
    sv.players["n_cells"][:] = L.cap_cells
    ids = rng.permutation(L.P * L.cap_cells) + 100
    for p in range(L.P):
        c = sv.cells[p]
        c["x"], c["y"] = rng.uniform(0, W, L.cap_cells), rng.uniform(0, W, L.cap_cells)
        c["mass"] = rng.choice([25, 100, 150, 200, 400, 2000], L.cap_cells)
        c["id"] = ids[p * L.cap_cells:(p + 1) * L.cap_cells]
    sv.players["bot_type"][L.A:] = rng.integers(0, 4, L.P - L.A)
    resp = sum(1 << p for p in range(1, L.P, 2))
    sv.hdr["respawned_lo"], sv.hdr["respawned_hi"] = resp & 0xFFFFFFFF, resp >> 32
    b.upload_state(0, sv)
    torch.cuda.synchronize()
    for size in (16, 48, 128, 256):
        pics = b.draw(i32([0, 1, 2, 3]), size, "agent").cpu().numpy()
        for a in range(4):
            assert np.array_equal(pics[a], oracle_draw(b.cfg, L, sv.blob, AGENT, a, size)), (size, a)
    redraw(b)  # the observation: pre_respawn 1
    check(b, instances=[0], what="crafted")
    assert (b.pixels()[1] == torch.tensor([0x2B, 0x2B, 0x33], dtype=torch.uint8, device="cuda")).all(), "respawned agent 1"


@pytest.mark.gpu
def test_refusals():
    from agarcl_b200 import _lib
    from agarcl_b200.batch import Batch
    L = _lib.lib()
    vp = C.c_void_p
    b, rng, pf, ps, _ = pixel_batch("c2", 32, N=2)
    d = np.zeros(4, np.float32)
    a = np.zeros(2, np.int32)
    lists = (C.c_uint8 * 256)()
    for rc, fn in ((L.agarcl_batch_step_host(b._h, d.ctypes.data_as(vp), a.ctypes.data_as(vp), None, None, None), "step_host"),
                   (L.agarcl_batch_step_mirror(b._h, d.ctypes.data_as(vp), a.ctypes.data_as(vp), None, None), "step_mirror"),
                   (L.agarcl_batch_step_lists(b._h, d.ctypes.data_as(vp), a.ctypes.data_as(vp), None, None, C.byref(lists)), "step_lists"),
                   (L.agarcl_batch_sync_mirror(b._h, None), "sync_mirror")):
        assert rc == -4, fn
        assert "pixel batch" in L.agarcl_last_error().decode(), fn
    with pytest.raises(_lib.AgarclError, match="final pictures"):
        b.final_pixels()
    g = Batch(make_cfg(n_instances=1, num_bots=0, num_viruses=0, num_pellets=50, arena_size=100))
    with pytest.raises(_lib.AgarclError, match="pixel_obs"):
        g.pixels()
    for kw in (dict(pixel_obs=40), dict(pixel_obs=64, num_frames=2), dict(pixel_obs=64, strict_reference=1),
               dict(pixel_obs=64, ram_obs=2)):
        with pytest.raises(_lib.AgarclError, match="pixel_obs"):
            Batch(make_cfg(**kw))


@pytest.mark.gpu
def test_python_layers():
    import torch
    from agarcl_b200 import BatchedGridEnvironment
    from agarcl_b200.gym_env import AgarioEnv, BatchedAgarioEnv
    env = BatchedAgarioEnv(4, obs_type="pixels", pixel_size=64, final_obs=True, num_agents=2, num_bots=4, arena_size=300,
                           num_pellets=300, num_viruses=4, number_steps=6)
    env.seed(3)
    obs, _ = env.reset()
    assert obs.shape == (8, 64, 64, 3) and obs.dtype == torch.uint8 and obs.is_cuda
    b = env._env.batch
    check(b, obs, what="BatchedAgarioEnv reset")
    pool = env.snapshot_pool(4)
    env.save_states(pool, i32([0, 1, 2, 3]))
    saved = obs.clone()
    for t in range(7):
        obs, rew, done, trunc, info = env.step(torch.zeros((8, 2), device="cuda"), torch.zeros(8, dtype=torch.int32, device="cuda"))
        assert obs.shape == (8, 64, 64, 3) and obs.dtype == torch.uint8
        assert info["final_obs"].shape == (8, 64, 64, 3) and info["final_obs"].dtype == torch.uint8
    assert info["reset_mask"].any()  # the step limit of 6
    restored = env.restore_states(pool, i32([0, 1, 2, 3]))
    assert torch.equal(restored, saved)
    env.close()

    g = BatchedGridEnvironment(2, num_agents=1, num_bots=2, arena_size=200, num_pellets=100, num_viruses=2, pixel_obs=32)
    o = g.reset()
    assert o.shape == (2, 32, 32, 3) and o.dtype == torch.uint8
    o, _, _ = g.step(np.zeros((2, 2), np.float32), np.zeros(2, np.int32))
    assert o.shape == (2, 32, 32, 3)
    g.close()

    e = AgarioEnv(obs_type="pixels", pixel_size=48)
    assert e.observation_space.shape == (48, 48, 3) and np.dtype(e.observation_space.dtype) == np.uint8
    e.seed(1)
    o, _ = e.reset()
    assert isinstance(o, np.ndarray) and o.shape == (48, 48, 3) and o.dtype == np.uint8
    o, r, d, tr, info = e.step(([0.5, 0.5], 0))
    assert o.shape == (48, 48, 3)
    check(e._env._ensure(), what="AgarioEnv")
    e.close()
    m = AgarioEnv(obs_type="pixels", pixel_size=32, num_agents=3, num_bots=2)
    o, _ = m.reset()
    assert isinstance(o, list) and len(o) == 3 and all(x.shape == (32, 32, 3) and x.dtype == np.uint8 for x in o)
    m.close()
