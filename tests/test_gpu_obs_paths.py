"""-m gpu: every path that writes the grid observation, compared bit for bit with the oracle (oracle_step / oracle_obs).

The step has several implementations of the observation, chosen by dtype, grid size, channel count, num_frames,
strict_reference and AGARCL_FUSE_CLEAR (DESIGN.md section 3, "Which kernel writes the observation"):
  A        k_step finishes the whole int32 frame itself (obs_finish_warp<int32_t>); "A-lists": it also writes the host-mirror
           lists, "A-pack": the grid's record is too long for one warp store and k_pack makes the lists
  A16      the same for int16 (CAS on 32-bit words, saturating at 32767)
  B / B'   k_step clears channels 1..C-1, k_obs (skip_zero) writes channel 0 and scatters: elementwise / 16-byte vector branch
  C        k_obs writes the whole frame
  D        several frames: one k_step per tick, k_obs for each rendered tick, a closing k_step
  E        strict_reference: the frame of the reference's frame-index arithmetic (quirk Q11)
  F        render(): k_obs on the current state, no tick in between
Every case names its path and checks it through launches_per_step(): the single fused kernel is k_step + k_order = 2 and
k_obs adds one; under step_mirror k_pack adds one more unless k_step wrote the lists.  State, rewards and dones are compared
on every step as well, so a frame cannot be right by accident of a diverged game.
"""
import numpy as np
import pytest

from _helpers import Oracle
from agarcl_b200 import OBS_I16, OBS_I32, make_cfg
from agarcl_b200._abi import compare_states
from agarcl_b200._lib import AgarclError
from agarcl_b200.batch import Batch
from gpu_parity_lib import run_parity

pytestmark = pytest.mark.gpu

# small arena, every channel populated: pellets, viruses, bots of every size, agents split (boost)
BASE = dict(num_agents=2, num_bots=8, arena_size=300, num_pellets=300, num_viruses=10, cap_foods=2048)
SEEDS = [71, 72]


def clip16(o):
    """the int16 reference: every scatter operation is monotone, so saturating each update = clipping the int32 frame"""
    return np.clip(o, -32768, 32767)


def mirror_allowed(G, dtype):
    return (G * G * (2 if dtype == OBS_I16 else 4)) % 16 == 0


# path -> (launches of Batch.step, k_step writes the host lists)
PATHS = {"A-lists": (2, True), "A-pack": (2, False), "A16-lists": (2, True), "A16-pack": (2, False),
         "B": (3, False), "B'": (3, False), "C": (3, False)}


def expect_launches(path, via):
    n, lists = PATHS[path]
    return n + (1 if via == "mirror" and not lists else 0)


def run_case(cfg_kwargs, path, via, steps=30, obs_every=3, launches=None, **kw):
    """run_parity through `via` and the check that the case took `path` (launches: the expected count, when not a PATHS entry)"""
    dtype = cfg_kwargs.get("obs_dtype", OBS_I32)
    if dtype == OBS_I16:
        kw.setdefault("obs_ref", clip16)
    stats = run_parity(cfg_kwargs, seeds=SEEDS, steps=steps, obs_every=obs_every, via=via, **kw)
    want = launches if launches is not None else expect_launches(path, via)
    assert stats["launches"] == [want], f"{path} via {via}: launches {stats['launches']}, want {want} -- the case took another path"
    return stats


def assert_lists_refused(cfg_kwargs, match):
    """step_lists refuses this configuration, and a refused call has not stepped anything"""
    b = Batch(make_cfg(n_instances=2, **cfg_kwargs))
    b.seed(9)
    b.reset()
    before = [b.download_state(i) for i in range(b.N)]
    NA = b.N * b.A
    with pytest.raises(AgarclError, match=match):
        b.step_lists(np.zeros((NA, 2), np.float32), np.zeros(NA, np.int32))
    for i in range(b.N):
        d = compare_states(before[i], b.download_state(i))
        assert not d, f"a refused step_lists changed instance {i}: {d[:4]}"
    b.close()


def assert_mirror_refused(cfg_kwargs):
    b = Batch(make_cfg(n_instances=2, **cfg_kwargs))
    b.seed(9)
    b.reset()
    with pytest.raises(AgarclError, match="multiples of 16 bytes"):
        b.mirror()
    b.close()


# grid size -> path, one frame, default knobs
# (the row of y masks lives in the collision scratch: 1824 B unless the pellet hash is larger, so int32 grids above 456 and int16
# grids above 912 take k_obs even below the 2560 B tile -- G 640 / 1024 reach the tile edge with AGARCL_HASH_PER_CELL, below)
I32_GRIDS = {1: "C", 2: "B", 3: "C", 4: "A-lists", 33: "C", 42: "B", 84: "A-lists", 100: "A-lists", 127: "C", 416: "A-lists",
             420: "A-pack", 452: "A-pack", 456: "A-pack", 460: "B'", 640: "B'", 644: "B'", 1024: "B'"}
I16_GRIDS = {4: "B", 8: "A16-lists", 12: "B", 36: "B", 84: "B", 128: "A16-lists", 420: "B", 912: "A16-pack", 920: "B'", 1024: "B'"}
GRID_CASES = [(G, OBS_I32, p) for G, p in I32_GRIDS.items()] + [(G, OBS_I16, p) for G, p in I16_GRIDS.items()]


def _grid_id(c):
    return f"{'i16' if c[1] == OBS_I16 else 'i32'}-G{c[0]}-{c[2]}"


def _run_grid(cfg_kwargs, path, via):
    G, dtype = cfg_kwargs["grid_size"], cfg_kwargs.get("obs_dtype", OBS_I32)
    big = G >= 400
    if via == "mirror" and not mirror_allowed(G, dtype):
        return assert_mirror_refused(cfg_kwargs)
    if via == "lists" and not PATHS[path][1]:
        return assert_lists_refused(cfg_kwargs, "not finished by the step kernel")
    # (G 1024: 32 MiB per int32 image, four images; the large grids compare every fifth step)
    run_case(cfg_kwargs, path, via, steps=20 if big else 30, obs_every=5 if big else 3, boost=60)


@pytest.mark.parametrize("via", ["step", "mirror", "lists"])
@pytest.mark.parametrize("case", GRID_CASES, ids=_grid_id)
def test_grid_sizes_match_oracle(case, via):
    """Every grid size class of the table: the fused finish with whole and partial mask words, the record-size edge
    (G 416 = 32 record words; 420, 452: k_pack), the scratch edge (456 / 460), both k_obs branches, and odd grids.  G 4
    (int32) and 8 (int16) are the smallest fused grids: one grid cell spans 25-75 world units, the pellet window's slack
    matters."""
    G, dtype, path = case
    _run_grid(dict(BASE, grid_size=G, obs_dtype=dtype), path, via)


def test_int16_odd_channel_count_shares_words_across_images():
    """observe_cells=False: C = 7, so with int16 the last element of one image and the first of the next share a 32-bit
    word, and neighbouring k_obs CTAs update it with CAS (path C: G 33, the plane is not a 16-byte multiple)."""
    cfg = dict(BASE, grid_size=33, obs_dtype=OBS_I16, observe_cells=False)
    run_case(cfg, "C", "step", boost=60)
    assert_mirror_refused(cfg)


CHANNEL_SETS = [dict(observe_pellets=bool(m & 1), observe_viruses=bool(m & 2), observe_cells=bool(m & 4), observe_others=bool(m & 8))
                for m in range(16)]


@pytest.mark.parametrize("G", [64, 33])
@pytest.mark.parametrize("m", range(16), ids=lambda m: f"ch{m:04b}")
def test_channel_subsets_match_oracle(m, G):
    """All 16 combinations of observe_{pellets, viruses, cells, others}: at G 64 the fused finish (C = 1, nothing but the
    out-of-bounds mask, takes k_obs alone) through the host mirror, at G 33 k_obs alone."""
    flags = CHANNEL_SETS[m]
    path = "C" if G == 33 or m == 0 else "A-lists"
    run_case(dict(BASE, grid_size=G, **flags), path, "mirror" if G == 64 else "step", steps=20, boost=200)


# (ticks_per_step, num_frames, grid, dtype) -> launches of one step: path D = tps one-tick k_steps, k_obs for each of the last
# num_frames ticks, the closing k_step; path E (strict_reference) = k_step + k_obs of the one frame
FRAME_CASES = {
    "D-tps4-frames4": (dict(ticks_per_step=4, num_frames=4, grid_size=40), 4 + 4 + 1),
    "D-tps2-frames4-memset": (dict(ticks_per_step=2, num_frames=4, grid_size=40), 2 + 2 + 1),
    "D-tps4-frames3": (dict(ticks_per_step=4, num_frames=3, grid_size=40), 4 + 3 + 1),
    "D-i16-frames2": (dict(ticks_per_step=4, num_frames=2, grid_size=36, obs_dtype=OBS_I16), 4 + 2 + 1),
    "E-strict-tps1-frames1": (dict(ticks_per_step=1, num_frames=1, grid_size=40, strict_reference=True), 2),
    "E-strict-tps2-frames2": (dict(ticks_per_step=2, num_frames=2, grid_size=40, strict_reference=True), 2),
}


@pytest.mark.parametrize("via", ["step", "mirror", "lists"])
@pytest.mark.parametrize("name", list(FRAME_CASES))
def test_frames_and_strict_reference_match_oracle(name, via):
    kw, launches = FRAME_CASES[name]
    cfg = dict(BASE, **kw)
    if via == "lists":
        return assert_lists_refused(cfg, "single fused step kernel")
    run_case(cfg, name[0], via, launches=launches + (1 if via == "mirror" else 0), steps=25, obs_every=2, boost=60)


@pytest.mark.parametrize("via", ["step", "mirror", "lists"])
def test_forty_agents_match_oracle(via):
    """agent indices >= 32 in the fused finish, in the list slots (pos * A + a) and in the action prefetch"""
    run_case(dict(num_agents=40, num_bots=0, arena_size=300, num_pellets=300, num_viruses=10, cap_foods=2048, grid_size=32),
             "A-lists", via, steps=20)


# AGARCL_* knob -> (observation settings, path)
KNOB_CASES = {
    "FUSE_CLEAR=0": ({"AGARCL_FUSE_CLEAR": "0"}, dict(grid_size=64), "C"),
    "FUSE_CLEAR=1": ({"AGARCL_FUSE_CLEAR": "1"}, dict(grid_size=64), "B'"),
    "ZERO_CHUNKS=1": ({"AGARCL_ZERO_CHUNKS": "1"}, dict(grid_size=64), "A-lists"),
    "ZERO_CHUNKS=3": ({"AGARCL_ZERO_CHUNKS": "3"}, dict(grid_size=64), "A-lists"),
    "ZERO_CHUNKS=1000": ({"AGARCL_ZERO_CHUNKS": "1000"}, dict(grid_size=64), "A-lists"),
    "HASH_PER_CELL=0.05-G64": ({"AGARCL_HASH_PER_CELL": "0.05"}, dict(grid_size=64), "A-lists"),  # HG clamps to 64
    "HASH_PER_CELL=1000-G64": ({"AGARCL_HASH_PER_CELL": "1000"}, dict(grid_size=64), "A-lists"),  # HG clamps to 4
    "HASH_PER_CELL=0.05-G4": ({"AGARCL_HASH_PER_CELL": "0.05"}, dict(grid_size=4), "A-lists"),
    "HASH_PER_CELL=1000-G4": ({"AGARCL_HASH_PER_CELL": "1000"}, dict(grid_size=4), "A-lists"),
    # HG 64: a 16 KB hash-build scratch holds the row of y masks, so the 2560 B tile is the edge of the fused finish
    "HASH_PER_CELL=0.05-G640": ({"AGARCL_HASH_PER_CELL": "0.05"}, dict(grid_size=640), "A-pack"),
    "HASH_PER_CELL=0.05-G644": ({"AGARCL_HASH_PER_CELL": "0.05"}, dict(grid_size=644), "B'"),
    "HASH_PER_CELL=0.05-i16-G1024": ({"AGARCL_HASH_PER_CELL": "0.05"}, dict(grid_size=1024, obs_dtype=OBS_I16), "A16-pack"),
}


@pytest.mark.parametrize("via", ["step", "mirror"])
@pytest.mark.parametrize("name", list(KNOB_CASES))
def test_knobs_match_oracle(name, via, monkeypatch):
    """The A/B knobs each select another observation path (FUSE_CLEAR), split the fused clear differently (ZERO_CHUNKS) or
    change the pellet window of the finish and the bots' pellet search (HASH_PER_CELL): the tick parity matters there too."""
    env, obs, path = KNOB_CASES[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    big = obs["grid_size"] >= 400
    run_case(dict(BASE, **obs), path, via, steps=20 if big else 30, obs_every=5 if big else 3, boost=60)


def test_refused_step_lists_leaves_the_games_unchanged():
    """G 420: an image's record is 34 words, k_step cannot write it, so step_lists is refused -- before anything runs."""
    assert_lists_refused(dict(BASE, grid_size=420), "not finished by the step kernel")


# ---- crafted states, rendered by k_obs (path F) and compared with oracle_obs

W = 300.0


def _put(sv, p, x, y, masses):
    sv.players["n_cells"][p] = len(masses)
    for k, m in enumerate(masses):
        sv.cells[p][k]["x"] = np.float32(x)
        sv.cells[p][k]["y"] = np.float32(y)
        sv.cells[p][k]["mass"] = m


def _grid_borders(px, view, G):
    """world coordinates that fall exactly on grid-cell borders of the view (in the kernels' fp32 arithmetic)"""
    k = np.arange(G + 1, dtype=np.float32)
    return np.float32(px) + (k - np.float32(G / 2.0)) * np.float32(view) / np.float32(G)


def _scene(i, sv, G, rng):
    """instance i of the crafted batch (2 agents, 4 bots, 300 pellets, 400 viruses)"""
    npel, nvir = int(sv.hdr["n_pellets"]), int(sv.hdr["n_viruses"])
    assert npel == 300 and nvir == 400, (npel, nvir)
    pel, vir = sv.pellets, sv.viruses
    if i == 0:  # a dead agent (quirk Q20): NaN centroid, channel 0 all -1, nothing scattered
        sv.players["n_cells"][0] = 0
        _put(sv, 1, 150.0, 150.0, [50])
    elif i == 1:  # an agent at a corner and one on an edge; entities just outside the view truncate into row / column 0
        _put(sv, 0, 0.0, 0.0, [50])
        _put(sv, 1, W - 0.5, 150.0, [50])
        h = 50.0 + 100.0 / G + 2.0
        u = rng.uniform(0.0, 1.0, npel).astype(np.float32)
        pel["x"][:150] = np.clip(W - 0.5 - h + u[:150] * 4.0, 0, W)
        pel["y"][:150] = rng.uniform(100.0, 200.0, 150)
        pel["x"][150:] = rng.uniform(0.0, 60.0, 150)
        pel["y"][150:] = np.clip(50.0 - 2.0 + u[150:] * (h - 48.0), 0, W)
        vir["x"][:200] = np.clip(W - 0.5 - h + rng.uniform(0, 4, 200), 0, W)
        vir["y"][:200] = rng.uniform(90.0, 210.0, 200)
    elif i == 2:  # entities exactly on grid-cell borders of the view, and at x = W / y = W
        _put(sv, 0, 200.0, 200.0, [60])
        _put(sv, 1, 270.0, 270.0, [60])
        b0, b1 = _grid_borders(200.0, 120.0, G), _grid_borders(270.0, 120.0, G)
        pel["x"][:100] = rng.choice(b0, 100)
        pel["y"][:100] = rng.choice(b0, 100)
        pel["x"][100:200] = np.minimum(rng.choice(b1, 100), W)
        pel["y"][100:200] = np.minimum(rng.choice(b1, 100), W)
        pel["x"][200:250] = W
        pel["y"][200:250] = rng.uniform(220.0, W, 50)
        pel["y"][250:] = W
        pel["x"][250:] = rng.choice(np.minimum(b1, W), 50)
        vir["x"][:50] = W
        vir["y"][:50] = rng.choice(np.minimum(b1, W), 50)
    elif i == 3:  # 400 viruses on one point of the view: channel 4 sums past 40 000, channel 3 is the last writer
        _put(sv, 0, 150.0, 150.0, [50])
        _put(sv, 1, 100.0, 100.0, [50])
        vir["x"][:] = 160.0
        vir["y"][:] = 150.0
        vir["mass"][:] = 100
        vir["mass"][200] = 150
        vir["mass"][nvir - 1] = 137
        pel["x"][:] = 140.0
        pel["y"][:] = 150.0
    else:  # masses around the int16 limit sharing grid cells: own sum, min over non-zero and max of the others
        _put(sv, 0, 150.0, 150.0, [32766, 32767, 32768, 40000])
        _put(sv, 1, 180.0, 150.0, [32767, 32768])
        _put(sv, 2, 170.0, 150.0, [32766, 40000, 32768, 32767])
        _put(sv, 3, 170.0, 130.0, [32768, 40000])
        _put(sv, 4, 130.0, 140.0, [32767, 32768])
        _put(sv, 5, 120.0, 160.0, [40000])


@pytest.mark.parametrize("dtype", [OBS_I32, OBS_I16], ids=["i32", "i16"])
@pytest.mark.parametrize("G", [1, 33, 84, 128])
def test_render_crafted_states_matches_oracle(G, dtype):
    import torch
    n = 5
    cfg = make_cfg(n_instances=n, num_agents=2, num_bots=4, arena_size=int(W), num_pellets=300, num_viruses=400, grid_size=G,
                   obs_dtype=dtype)
    b = Batch(cfg)
    b.seed(17)
    b.reset()
    rng = np.random.default_rng(G)
    states = []
    for i in range(n):
        sv = b.download_state(i)
        _scene(i, sv, G, rng)
        b.upload_state(i, sv)
        states.append(sv)
    b.render()
    torch.cuda.synchronize()
    g = b.obs_tensor().cpu().numpy().reshape(n, b.A, -1, G, G)
    A = b.A
    for i, sv in enumerate(states):
        o = Oracle(cfg, b.layout)
        o.state = sv
        want = np.stack([o.obs(a) for a in range(A)])
        if i == 3:
            assert want[0][4].max() >= 40000 and (want[0][3] == 137).any()
        if i == 4:
            assert want[0][5].max() > 32767 and want[0][7].max() == 40000
        ref = clip16(want) if dtype == OBS_I16 else want
        for a in range(A):
            if not np.array_equal(g[i][a], ref[a]):
                bad = [(c, int((g[i][a][c] != ref[a][c]).sum())) for c in range(ref.shape[1]) if not np.array_equal(g[i][a][c], ref[a][c])]
                raise AssertionError(f"G {G} scene {i} agent {a}: (channel, #cells) differ {bad}")
    assert (g[0][0][0] == -1).all() and not g[0][0][1:].any(), "a dead agent sees only out-of-bounds"
    b.close()


def test_stacked_viruses_saturate_the_fused_int16_finish():
    """Path A16 (G 128 int16): 400 viruses on one point in the view, away from every player, stepped once by k_step and by
    the oracle from the same uploaded state; channel 4 (40 000+) saturates at 32767 inside FinOps<int16_t>."""
    peaks = []

    def stack(i, sv):
        assert int(sv.hdr["n_viruses"]) == 400
        px, py = float(sv.cells[0][0]["x"]), float(sv.cells[0][0]["y"])
        vx = px + 30.0 if px < 200.0 else px - 30.0
        sv.viruses["x"][:] = vx
        sv.viruses["y"][:] = py
        sv.viruses["mass"][:] = 100
        sv.viruses["mass"][399] = 121

    def ref(o):
        peaks.append(int(o[:, 4].max()))
        return clip16(o)

    run_case(dict(num_agents=1, num_bots=0, arena_size=300, num_pellets=100, num_viruses=400, grid_size=128, obs_dtype=OBS_I16),
             "A16-lists", "step", steps=1, obs_every=1, edit=stack, obs_ref=ref)
    assert peaks and min(peaks) >= 40000, peaks
