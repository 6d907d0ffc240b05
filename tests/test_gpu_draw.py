"""Pictures of game states on the device (agarcl_batch_draw, draw_kernel.cu): byte-exact against oracle_draw on downloaded
blobs across configurations, ages, views and sizes, a crafted maximal state, source indexing, no effect on the game, no host
wait, the refusals and the Python layers."""
import ctypes as C

import numpy as np
import pytest

from _helpers import AGENT, ARENA, RGB, oracle_draw
from agarcl_b200 import make_cfg
from gpu_parity_lib import aged_batch, device_record, i32, step_random

CASES = ["c1", "c2", "c3", "c4_four_agents", "c5", "mode1", "mode8", "mixed_tasks", "int16", "ram_obs2", "strict_reference",
         "mt19937"]


def _check(b, view, size, src=None):
    """device pictures of src (None: every source) against oracle_draw on the downloaded blobs"""
    import torch
    pics = b.draw(None if src is None else i32(src), size, "agent" if view == AGENT else "arena")
    torch.cuda.synchronize()
    pics = pics.cpu().numpy()
    n_src = b.N * (b.A if view == AGENT else 1)
    src = list(range(n_src)) if src is None else list(src)
    blobs = {}
    for k, s in enumerate(src):
        if not 0 <= s < n_src:
            assert not pics[k].any(), f"source {s} out of range: not all zero"
            continue
        i, a = (s // b.A, s % b.A) if view == AGENT else (s, 0)
        if i not in blobs:
            blobs[i] = b.download_state(i).blob
        exp = oracle_draw(b.cfg, b.layout, blobs[i], view, a, size)
        if not np.array_equal(pics[k], exp):
            bad = np.argwhere(np.any(pics[k] != exp, axis=-1))
            raise AssertionError(f"view {view} size {size} source {s}: {len(bad)} pixels differ, first {bad[:4].tolist()}: "
                                 f"{pics[k][tuple(bad[0])]} vs {exp[tuple(bad[0])]}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_pictures_match_oracle(name):
    """both views at 16 and 128 for every source at ages 0, 1 and 250; 512 and 2048 on a few pictures of the aged state"""
    b, rng, p_feed, p_split = aged_batch(name)
    for age, more in ((0, 0), (1, 1), (250, 249)):
        step_random(b, rng, p_feed, p_split, more)
        for view in (ARENA, AGENT):
            for size in (16, 128):
                _check(b, view, size)
    _check(b, ARENA, 512, [0, 3])
    _check(b, AGENT, 512, [b.N * b.A - 1])
    if name in ("c2", "c4_four_agents"):
        _check(b, ARENA, 2048, [1])
        _check(b, AGENT, 2048, [0])
    if name == "c4_four_agents":  # the agents did split
        assert max(int(b.download_state(i).players["n_cells"][:b.A].max()) for i in range(b.N)) > 1
    b.close()


@pytest.mark.gpu
def test_crafted_maximal_state():
    """64 players x 32 cells and full pellet, virus and food capacities: more than one pass of every culled list"""
    from agarcl_b200.batch import Batch
    import torch
    b = Batch(make_cfg(n_instances=2, num_agents=4, num_bots=60, num_viruses=60, num_pellets=1500, arena_size=600))
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
        c["mass"] = rng.choice([25, 100, 150, 200, 400, 2000], L.cap_cells)  # many equal masses: the kind and id decide
        c["id"] = ids[p * L.cap_cells:(p + 1) * L.cap_cells]
    sv.players["bot_type"][L.A:] = rng.integers(0, 4, L.P - L.A)
    b.upload_state(0, sv)
    torch.cuda.synchronize()
    for size in (16, 32, 128, 512):
        _check(b, ARENA, size, [0])
    for size in (16, 128):
        _check(b, AGENT, size, [0, 1, 2, 3])
    b.close()


@pytest.mark.gpu
def test_source_indexing():
    """d_src NULL draws every source in order; duplicates repeat a picture; out-of-range entries give zeros"""
    import torch
    b, rng, pf, ps = aged_batch("c4_four_agents", N=3)
    step_random(b, rng, pf, ps, 20)
    for view, n_src in (("arena", b.N), ("agent", b.N * b.A)):
        every = b.draw(None, 64, view)
        assert every.shape == (n_src, 64, 64, 3)
        src = [2, 2, -1, n_src, 0, n_src - 1, -(1 << 31), (1 << 31) - 1]
        some = b.draw(i32(src), 64, view)
        torch.cuda.synchronize()
        every, some = every.cpu().numpy(), some.cpu().numpy()
        for k, s in enumerate(src):
            if 0 <= s < n_src:
                assert np.array_equal(some[k], every[s])
            else:
                assert not some[k].any()
    _check(b, ARENA, 64, [2, 2, -1, 3, 0])
    _check(b, AGENT, 64, [5, -1, 12, 11])


@pytest.mark.gpu
def test_drawing_changes_nothing():
    """state blobs, observation, rewards, dones, ram records, episode buffers, final observations and ram records and the host
    mirror are bitwise the same after drawing, and the following steps equal those of a twin batch that never drew"""
    import torch
    from agarcl_b200.batch import Batch
    cfg = make_cfg(n_instances=8, ram_obs=1, num_bots=6, arena_size=300, num_pellets=300, num_viruses=4)
    twins = [Batch(cfg), Batch(cfg)]
    for b in twins:
        b.seed(42)
        b.reset()
        b.set_autoreset(30, keep_final_obs=True)
        b.sync_mirror()
    rng = np.random.default_rng(0)
    for t in range(60):
        dxdy = rng.uniform(-1, 1, (cfg.n_instances, 2)).astype(np.float32)
        act = rng.integers(0, 3, cfg.n_instances).astype(np.int32)
        for b in twins:
            b.set_actions(dxdy, act)
            b.step_autoreset()
            b.sync_mirror()
        if t % 10 == 3:
            before = device_record(twins[0])
            for view in ("arena", "agent"):
                for size in (16, 144, 512):
                    twins[0].draw(None, size, view)
            twins[0].draw(i32([0, -5, 99]), 32, "arena")
            after = device_record(twins[0])
            for k in before:
                assert np.array_equal(before[k], after[k]), f"step {t}: draw changed {k}"
        a, c = device_record(twins[0]), device_record(twins[1])
        for k in a:
            assert np.array_equal(a[k], c[k]), f"step {t}: {k} differs from the twin that never drew"
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_no_host_wait_graph_capture_and_interleaved_steps():
    """after one warm-up the call is captured in a CUDA graph (capture fails on any synchronising call) and the replay gives
    the same bytes; interleaved with step_autoreset on one stream, every step gets its own picture"""
    import torch
    b, rng, pf, ps = aged_batch("c2", N=4)
    step_random(b, rng, pf, ps, 30)
    src = i32([3, 1, 0])
    s = torch.cuda.Stream()
    out = torch.zeros((3, 128, 128, 3), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        b.draw(src, 128, "arena", out=out, stream=s.cuda_stream)  # warm-up
    s.synchronize()
    eager = out.clone()
    out.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        b.draw(src, 128, "arena", out=out, stream=s.cuda_stream)
    torch.cuda.synchronize()
    assert not out.any()  # captured, not run
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)

    b.set_autoreset(40)
    T = 12
    video = torch.zeros((T, b.N, 64, 64, 3), dtype=torch.uint8, device="cuda")
    blobs = []
    for t in range(T):
        b.set_actions(*[x for x in (rng.uniform(-1, 1, (b.N, 2)).astype(np.float32), rng.integers(0, 3, b.N).astype(np.int32))])
        b.step_autoreset()
        b.draw(None, 64, "arena", out=video[t])
        blobs.append([b.download_state(i).blob for i in range(b.N)])  # (waits: test only)
    video = video.cpu().numpy()
    for t in range(T):
        for i in range(b.N):
            assert np.array_equal(video[t, i], oracle_draw(b.cfg, b.layout, blobs[t][i], ARENA, 0, 64)), f"step {t} instance {i}"


@pytest.mark.gpu
def test_refusals_leave_the_output_untouched():
    import torch
    from agarcl_b200 import _lib
    from agarcl_b200.batch import Batch
    L = _lib.lib()
    vp = C.c_void_p
    cfg = make_cfg(n_instances=2, num_bots=2, arena_size=200, num_pellets=100, num_viruses=2)
    fresh = Batch(cfg)
    out = torch.full((2, 64, 64, 3), 0xAB, dtype=torch.uint8, device="cuda")

    def refused(b, view, size, n, ptr, text, rc=-1):
        got = L.agarcl_batch_draw(b._h, view, size, None, n, vp(ptr), None)
        assert got == rc, (got, text)
        assert text in L.agarcl_last_error().decode(), L.agarcl_last_error().decode()
        torch.cuda.synchronize()
        assert bool((out == 0xAB).all()), f"{text}: output written"

    refused(fresh, 0, 64, 2, out.data_ptr(), "before reset", rc=-4)
    b = Batch(cfg)
    b.seed(1)
    b.reset()
    refused(b, 2, 64, 2, out.data_ptr(), "unknown view")
    refused(b, -1, 64, 2, out.data_ptr(), "unknown view")
    for size in (0, 8, 24, 2064, 4096, -16):
        refused(b, 0, size, 2, out.data_ptr(), "multiple of 16")
    refused(b, 0, 64, -1, out.data_ptr(), "n must be >= 0")
    refused(b, 0, 64, 2, 0, "null output")
    refused(b, 0, 64, 1, out.data_ptr() + 8, "16-byte aligned")
    host = np.zeros(64 * 64 * 3 + 64, np.uint8)
    hp = (host.ctypes.data + 15) & ~15
    refused(b, 0, 64, 1, hp, "device memory")
    assert not host.any()
    pinned = torch.zeros(64 * 64 * 3, dtype=torch.uint8).pin_memory()
    refused(b, 0, 64, 1, pinned.data_ptr(), "device memory")
    assert not pinned.any()
    with pytest.raises(_lib.AgarclError, match="unknown view"):
        b.draw(None, 64, "screen")
    with pytest.raises(_lib.AgarclError, match="out must be"):
        b.draw(None, 64, "arena", out=out[:1])
    with pytest.raises(_lib.AgarclError, match="int32"):
        b.draw(torch.zeros(2, dtype=torch.int64, device="cuda"), 64)
    assert bool((out == 0xAB).all())
    assert L.agarcl_batch_draw(b._h, 0, 64, None, 0, vp(out.data_ptr()), None) == 0  # n = 0: nothing
    torch.cuda.synchronize()
    assert bool((out == 0xAB).all())


@pytest.mark.gpu
def test_python_layers():
    """BatchedAgarioEnv.render and AgarioEnv(render_mode="rgb_array").render() are Batch.draw; the other render modes and the
    reference-named render() / get_frame() still raise"""
    import torch
    from agarcl_b200 import GridEnvironment
    from agarcl_b200.gym_env import AgarioEnv, BatchedAgarioEnv
    env = BatchedAgarioEnv(4, num_agents=2, num_bots=4, arena_size=300, num_pellets=300, num_viruses=4)
    env.seed(3)
    env.reset()
    for _ in range(5):
        env.step(torch.zeros((8, 2), device="cuda"), torch.zeros(8, dtype=torch.int32, device="cuda"))
    b = env._env.batch
    pics = env.render()
    assert pics.shape == (4, 256, 256, 3) and pics.is_cuda
    assert torch.equal(pics, b.draw(None, 256, "arena"))
    ids = torch.tensor([2, 0], dtype=torch.int64, device="cuda")
    agents = env.render(ids, size=96, view="agent")
    assert torch.equal(agents, b.draw(i32([4, 5, 0, 1]), 96, "agent"))
    buf = torch.empty((2, 64, 64, 3), dtype=torch.uint8, device="cuda")
    assert env.render(ids, size=64, out=buf).data_ptr() == buf.data_ptr()
    assert torch.equal(buf, b.draw(i32([2, 0]), 64))
    env.close()

    e = AgarioEnv(render_mode="rgb_array", render_size=128)
    e.seed(1)
    e.reset()
    e.step(([0.5, 0.5], 0))
    pic = e.render()
    assert isinstance(pic, np.ndarray) and pic.shape == (128, 128, 3) and pic.dtype == np.uint8
    assert np.array_equal(pic, e._env._ensure().draw(None, 128, "arena").cpu().numpy()[0])
    assert np.array_equal(pic, oracle_draw(e._env._ensure().cfg, e._env._ensure().layout, e._env._ensure().download_state(0).blob,
                                           ARENA, 0, 128))
    e.close()
    m = AgarioEnv(render_mode="rgb_array", render_size=64, render_view="agent", num_agents=3, num_bots=2)
    m.reset()
    assert m.render().shape == (3, 64, 64, 3)
    m.close()
    for mode in (None, "human"):
        with pytest.raises(RuntimeError, match="OpenGL"):
            AgarioEnv(render_mode=mode).render()
    g = GridEnvironment(1, 4, 300, True, 100, 0, 0)
    for f in (g.render, g.get_frame):
        with pytest.raises(RuntimeError, match="OpenGL"):
            f()
    with pytest.raises(ValueError):
        AgarioEnv(render_mode="rgb_array", render_view="top")
    assert RGB["OUT"] != RGB["BACKGROUND"]
