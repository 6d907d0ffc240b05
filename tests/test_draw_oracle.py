"""Pictures of game states (include/agarcl_b200.h, agarcl_batch_draw), pinned through their CPU restatement oracle_draw
(tests/draw_oracle.c): the disc test against a numpy fp32 evaluation, the draw order, the agent view's tie to observation
channel 0 (of the oracle port), the one-pixel floor and the absent players of a mixed-task layout.  CPU only."""
import numpy as np
import pytest

from _helpers import AGENT, ARENA, RGB, aged_oracle, oracle_draw, oracle_layout
from agarcl_b200._abi import StateView, make_cfg, task_bits


def is_color(pic, rgb):
    return np.all(pic == np.asarray(rgb, np.uint8), axis=-1)


def radius(m):
    return np.float32(np.sqrt(np.float64(m) / np.pi))


def arena_coords(W, S):
    return ((np.arange(S, dtype=np.float32) + np.float32(0.5)) * np.float32(W)) / np.float32(S)


def disc(xs, ys, ex, ey, R):
    """(inside, border) masks [S, S] of the fp32 disc test, rows y and columns x"""
    dx = xs[None, :] - np.float32(ex)
    dy = ys[:, None] - np.float32(ey)
    d2 = dx * dx + dy * dy
    R = np.float32(R)
    b = np.float32(0.85) * R
    return d2 <= R * R, d2 > b * b


def _empty_state(**kw):
    cfg = make_cfg(**kw)
    L = oracle_layout(cfg)
    return cfg, L, StateView(L)


def test_single_cell_pellet_virus_against_numpy():
    """one cell, one pellet and one virus in the arena view: each disc is the numpy fp32 disc test with the one-pixel floor,
    borders included, and every other pixel is background"""
    S, W = 64, 100
    cfg, L, sv = _empty_state(num_bots=0, num_viruses=1, num_pellets=1, arena_size=W)
    sv.hdr["n_pellets"], sv.hdr["n_viruses"], sv.hdr["n_foods"] = 1, 1, 0
    sv.players["n_cells"][0] = 1
    c = sv.cells[0][0]
    c["x"], c["y"], c["mass"], c["id"] = 30.25, 40.5, 100, 1
    sv.pellets[0] = (70.0, 20.0)
    v = sv.viruses[0]
    v["x"], v["y"], v["mass"] = 72.0, 70.0, 150
    pic = oracle_draw(cfg, L, sv.blob, ARENA, 0, S)
    xs = ys = arena_coords(W, S)
    px = np.float32(W) / np.float32(S)
    cell_in, cell_b = disc(xs, ys, 30.25, 40.5, max(radius(100), px))
    pel_in, _ = disc(xs, ys, 70.0, 20.0, max(radius(1), px))
    vir_in, vir_b = disc(xs, ys, 72.0, 70.0, max(radius(150), px))
    assert pel_in.sum() >= 1 and not (cell_in & pel_in).any() and not (cell_in & vir_in).any() and not (pel_in & vir_in).any()
    exp = np.empty((S, S, 3), np.uint8)
    exp[:] = RGB["BACKGROUND"]
    exp[pel_in] = RGB["PELLET"]
    agent = np.asarray(RGB["AGENTS"][0])
    exp[cell_in & ~cell_b] = agent
    exp[cell_in & cell_b] = agent * 3 // 4
    exp[vir_in & ~vir_b] = RGB["VIRUS"]
    exp[vir_in & vir_b] = RGB["VIRUS_BORDER"]
    assert np.array_equal(pic, exp)
    assert (cell_in & cell_b).any() and (cell_in & ~cell_b).any() and (vir_in & vir_b).any()


def test_draw_order_mass_kind_id():
    """overlapping cells of different mass, a virus of a mass between them, and equal-mass ties: painted by (mass, kind, id)
    ascending, a virus under a cell of its mass, the lower id under the higher"""
    S, W = 128, 100
    cfg, L, sv = _empty_state(num_bots=3, num_viruses=1, num_pellets=1, arena_size=W)
    sv.hdr["n_pellets"], sv.hdr["n_viruses"], sv.hdr["n_foods"] = 0, 1, 0
    # (player, x, y, mass, id)
    cells = [(0, 50.0, 50.0, 400, 7), (1, 62.0, 50.0, 200, 3), (2, 62.0, 62.0, 300, 9), (3, 38.0, 62.0, 300, 4)]
    for p, x, y, m, i in cells:
        sv.players["n_cells"][p] = 1
        c = sv.cells[p][0]
        c["x"], c["y"], c["mass"], c["id"] = x, y, m, i
    sv.players["bot_type"][1:4] = [0, 1, 2]
    v = sv.viruses[0]
    v["x"], v["y"], v["mass"] = 50.0, 64.0, 300
    pic = oracle_draw(cfg, L, sv.blob, ARENA, 0, S)
    xs = ys = arena_coords(W, S)
    px = np.float32(W) / np.float32(S)
    ents = [((m, 1, i), x, y, RGB["AGENTS"][0] if p == 0 else RGB["BOTS"][p - 1], None) for p, x, y, m, i in cells]
    ents.append(((300, 0, 0), 50.0, 64.0, RGB["VIRUS"], RGB["VIRUS_BORDER"]))
    exp = np.empty((S, S, 3), np.uint8)
    exp[:] = RGB["BACKGROUND"]
    for key, x, y, col, border in sorted(ents, key=lambda e: e[0]):
        inside, b = disc(xs, ys, x, y, max(radius(key[0]), px))
        border = np.asarray(col) * 3 // 4 if border is None else border
        exp[inside & ~b] = col
        exp[inside & b] = border
    assert np.array_equal(pic, exp)
    # every entity shows, and the tie is decided: at the middle of the virus and the cell of its mass, the cell
    mid_r, mid_c = int(np.argmin(np.abs(ys - 63.0))), int(np.argmin(np.abs(xs - 44.0)))
    assert tuple(pic[mid_r, mid_c]) in (RGB["BOTS"][2], tuple(np.asarray(RGB["BOTS"][2]) * 3 // 4))
    assert is_color(pic, RGB["AGENTS"][0]).any() and is_color(pic, RGB["VIRUS"]).any()
    for t in range(3):
        assert is_color(pic, RGB["BOTS"][t]).any()


AGED = {
    "c2": (dict(), None),
    "c4": (dict(num_agents=4, num_bots=8, cap_foods=2048), 1000),
    "mode1": (dict(mode_number=1, num_bots=0), None),
}


@pytest.mark.parametrize("name", list(AGED))
def test_agent_view_out_of_arena_is_observation_channel0(name):
    """agent view at S = G on aged states: the out-of-arena pixels are exactly the -1 elements of channel 0, transposed"""
    kw, boost = AGED[name]
    checked = 0
    for seed in (3, 4, 5):
        o = aged_oracle(kw, seed, 40, boost)
        if int(o.state.hdr["respawned_lo"]) or int(o.state.hdr["respawned_hi"]):
            continue  # (the observation of the step shows respawned players dead)
        G = o.cfg.grid_size
        for a in range(o.L.A):
            pic = oracle_draw(o.cfg, o.L, o.state.blob, AGENT, a, G)
            out = is_color(pic, RGB["OUT"])
            assert np.array_equal(out, o.obs(a)[0].T == -1), f"{name} seed {seed} agent {a}"
            checked += 1
    assert checked


def test_agent_view_of_dead_agent_is_all_out_of_arena():
    o = aged_oracle(dict(num_agents=2, num_bots=4), 7, 5)
    o.state.players["n_cells"][1] = 0
    pic = oracle_draw(o.cfg, o.L, o.state.blob, AGENT, 1, 64)
    assert is_color(pic, RGB["OUT"]).all()
    assert (o.obs(1)[0] == -1).all()  # quirk Q20: the observation agrees


def test_one_pixel_floor_keeps_pellets_visible():
    """a 64-pixel picture of a 2000-unit arena: pixels are 31 units apart and a pellet's radius is 0.56, drawn at one pixel"""
    o = aged_oracle(dict(arena_size=2000, num_pellets=4000, num_viruses=50, cap_viruses=128), 9, 0)
    pic = oracle_draw(o.cfg, o.L, o.state.blob, ARENA, 0, 64)
    assert is_color(pic, RGB["PELLET"]).sum() > 64 * 64 // 4


def test_absent_players_draw_nothing():
    """mixed-task layout, an instance of mode 1 (no bot): the absent bot's slots hold stale cells, n_cells 0 -- nothing of
    them is drawn"""
    from agarcl_b200 import _lib
    cfg = make_cfg(mode_number=1, num_bots=0, task_modes=task_bits([1, 7]), arena_size=200, num_pellets=100, num_viruses=5)
    L = _lib.make_layout(cfg)
    assert L.P == 2
    sv = StateView(L)
    rng = np.random.default_rng(0)
    sv.hdr["n_pellets"], sv.hdr["n_viruses"] = 50, 5
    sv.pellets[:50] = [tuple(p) for p in rng.uniform(0, 200, (50, 2)).astype(np.float32)]
    for k in range(5):
        sv.viruses[k]["x"], sv.viruses[k]["y"], sv.viruses[k]["mass"] = *rng.uniform(0, 200, 2), 100
    sv.players["n_cells"][0] = 1
    sv.cells[0][0]["x"], sv.cells[0][0]["y"], sv.cells[0][0]["mass"], sv.cells[0][0]["id"] = 100, 100, 50, 1
    clean = sv.blob.copy()
    sv.players["bot_type"][1] = 0
    for i in range(8):  # stale cells of the absent player
        c = sv.cells[1][i]
        c["x"], c["y"], c["mass"], c["id"] = 20 + 20 * i, 50, 400, 10 + i
    for S in (64, 256):
        pic = oracle_draw(cfg, L, sv.blob, ARENA, 0, S)
        assert np.array_equal(pic, oracle_draw(cfg, L, clean, ARENA, 0, S))
        assert not is_color(pic, RGB["BOTS"][0]).any()
