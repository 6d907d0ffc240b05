"""Built-in bot policies for agents (include/agarcl_b200.h, agarcl_batch_bot_actions), pinned through oracle_bot_decide
(tests/bot_oracle.c: oracle.c's bot_take_action on a private copy of the blob) on crafted states: the nearest pellet against a
numpy fp32 brute force, the flee and chase triggers, no pellets, a dead agent, absent players of a mixed-task layout, and the
blob left untouched.  Also: k_bot_actions compiles for sm_100a without stack or spills.  CPU only."""
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from _helpers import aged_oracle, oracle_bot_decide, oracle_layout
from agarcl_b200._abi import (BOT_AGGRESSIVE, BOT_AGGRESSIVE_SHY, BOT_BAD_TYPE, BOT_DEAD, BOT_DECIDED, BOT_HUNGRY, BOT_HUNGRY_SHY,
                              BOT_NO_PELLET, BOT_SKIPPED, StateView, make_cfg, task_bits)

F = np.float32
TYPES = (BOT_HUNGRY, BOT_HUNGRY_SHY, BOT_AGGRESSIVE, BOT_AGGRESSIVE_SHY)


def _state(A=1, bots=3, pellets=64, arena=200, **kw):
    cfg = make_cfg(num_agents=A, num_bots=bots, num_viruses=0, num_pellets=pellets, arena_size=arena, **kw)
    L = oracle_layout(cfg)
    return cfg, L, StateView(L)


def _cell(sv, p, i, x, y, mass, cid=None):
    sv.players["n_cells"][p] = max(int(sv.players["n_cells"][p]), i + 1)
    c = sv.cells[p][i]
    c["x"], c["y"], c["mass"], c["id"] = x, y, mass, cid if cid is not None else 1 + p * 32 + i


def _loc(sv, p):
    """Player::x / y in fp32: sums in cell order, then one division"""
    n = int(sv.players["n_cells"][p])
    xs, ys, m = F(0), F(0), 0
    for i in range(n):
        c = sv.cells[p][i]
        xs = F(xs + F(c["x"]) * F(int(c["mass"])))
        ys = F(ys + F(c["y"]) * F(int(c["mass"])))
        m += int(c["mass"])
    with np.errstate(invalid="ignore", divide="ignore"):
        return F(xs / F(m)), F(ys / F(m))


def _pellets(sv, pts):
    sv.hdr["n_pellets"] = len(pts)
    for k, (x, y) in enumerate(pts):
        sv.pellets[k] = (x, y)


def _dxdy(target, loc):
    return np.array([F(F(target[0] - loc[0]) / F(10)), F(F(target[1] - loc[1]) / F(10))], np.float32)


def _expect(got, target, act, loc, status=BOT_DECIDED):
    dxdy, t, a, s = got
    assert s == status and a == act, (s, a)
    assert np.array_equal(t.view(np.uint32), np.asarray(target, np.float32).view(np.uint32)), (t, target)
    assert np.array_equal(dxdy.view(np.uint32), _dxdy(target, loc).view(np.uint32)), (dxdy, _dxdy(target, loc))


def test_nearest_pellet_is_numpy_first_minimum():
    """random pellets plus three at exactly the same distance and one closer than 0.01: the first strict minimum in array order
    of the fp32 distance among pellets with (double)d > 0.01"""
    cfg, L, sv = _state(bots=0, pellets=300)
    _cell(sv, 0, 0, 100.0, 100.0, 25)
    rng = np.random.default_rng(1)
    pts = rng.uniform(0, 200, (600, 2)).astype(np.float32)
    pts = [tuple(p) for p in pts[np.hypot(pts[:, 0] - 100, pts[:, 1] - 100) > 6][:300]]  # (none nearer than the three below)
    pts[7] = (100.005, 100.0)    # nearer than 0.01: never a target
    pts[40] = (104.0, 103.0)     # the three at distance 5: the first in array order wins
    pts[12] = (97.0, 96.0)
    pts[250] = (103.0, 104.0)
    _pellets(sv, pts)
    loc = _loc(sv, 0)
    px, py = np.array(pts, np.float32).T
    dx, dy = np.abs(loc[0] - px), np.abs(loc[1] - py)
    d = np.sqrt(dx * dx + dy * dy)
    assert d.dtype == np.float32
    ok = d.astype(np.float64) > 0.01
    best = d[ok].min()
    first = int(np.flatnonzero(ok & (d == best))[0])
    assert first == 12 and best == F(5) and not ok[7]
    for t in (BOT_HUNGRY, BOT_HUNGRY_SHY, BOT_AGGRESSIVE, BOT_AGGRESSIVE_SHY):
        _expect(oracle_bot_decide(cfg, L, sv.blob, 0, t), pts[first], 0, loc)
    # every pellet nearer than 0.01: target (0, 0)
    _pellets(sv, [(100.0, 100.0), (100.005, 100.0)])
    _expect(oracle_bot_decide(cfg, L, sv.blob, 0, BOT_HUNGRY), (0.0, 0.0), 0, loc)


@pytest.mark.parametrize("other_mass", [25, 400, 5000])
def test_flee_trigger_is_distance_below_25_whatever_the_masses(other_mass):
    cfg, L, sv = _state(bots=2)
    _cell(sv, 0, 0, 100.0, 100.0, 100)
    sv.players["action"][0] = 2
    _pellets(sv, [(60.0, 60.0), (150.0, 140.0)])
    loc = _loc(sv, 0)
    pellet = (60.0, 60.0)
    for x, flees in ((124.99, True), (125.0, False), (75.01, True)):
        _cell(sv, 1, 0, x, 100.0, other_mass)
        away = (F(loc[0] - F(F(x) - loc[0])), F(loc[1] - F(F(100.0) - loc[1])))
        _expect(oracle_bot_decide(cfg, L, sv.blob, 0, BOT_HUNGRY_SHY), away if flees else pellet, 0, loc)
        # AggressiveShy flees first and leaves the action as it is
        got = oracle_bot_decide(cfg, L, sv.blob, 0, BOT_AGGRESSIVE_SHY)
        if flees:
            _expect(got, away, 2, loc)
        _expect(oracle_bot_decide(cfg, L, sv.blob, 0, BOT_HUNGRY), pellet, 0, loc)


def test_flee_takes_the_first_player_in_the_order():
    cfg, L, sv = _state(bots=3)
    _cell(sv, 0, 0, 100.0, 100.0, 100)
    _pellets(sv, [(60.0, 60.0)])
    spots = {1: (110.0, 100.0), 2: (100.0, 115.0), 3: (90.0, 90.0)}
    for p, (x, y) in spots.items():
        _cell(sv, p, 0, x, y, 50)
    loc = _loc(sv, 0)
    first = [p for p in L.order[:L.P] if p != 0][0]
    ox, oy = spots[first]
    _expect(oracle_bot_decide(cfg, L, sv.blob, 0, BOT_HUNGRY_SHY), (F(loc[0] - F(F(ox) - loc[0])), F(loc[1] - F(F(oy) - loc[1]))),
            0, loc)


def _chase_target(sv, o, big, loc):
    sx, sy, m = F(0), F(0), 0
    for i in range(int(sv.players["n_cells"][o])):
        c = sv.cells[o][i]
        cm = int(c["mass"])
        if big > 25 and float(big) > float(cm) * 1.1:
            sx, sy, m = F(sx + F(c["x"]) * F(cm)), F(sy + F(c["y"]) * F(cm)), m + cm
    return (F(loc[0] + F(F(sx / F(m)) - loc[0]) * F(3)), F(loc[1] + F(F(sy / F(m)) - loc[1]) * F(3)))


def test_chase_trigger_is_distance_20_with_something_edible():
    cfg, L, sv = _state(bots=1)
    _cell(sv, 0, 0, 100.0, 100.0, 60)
    _cell(sv, 0, 1, 102.0, 100.0, 100)  # the largest cell: it eats below 100 / 1.1
    sv.players["action"][0] = 1
    _pellets(sv, [(30.0, 170.0)])
    loc = _loc(sv, 0)
    # the other player: two edible cells and one that is too big, moved in steps of 2^-16 along x
    cells = [(0.0, 0.0, 40), (4.0, 2.0, 90), (-3.0, 1.0, 95)]

    def place(k):
        for i, (x, y, cm) in enumerate(cells):
            _cell(sv, 1, i, F(118.0 + x + k * 2.0 ** -16), F(100.0 + y), cm)
        ox, oy = _loc(sv, 1)
        dx, dy = abs(loc[0] - ox), abs(loc[1] - oy)
        return np.sqrt(F(dx * dx + dy * dy))

    edge = max(k for k in range(0, 400000, 512) if place(k) <= 20)
    while place(edge + 1) <= 20:
        edge += 1
    for k, chases in ((edge, True), (edge + 1, False), (-1_000_000, True)):
        d = place(k)
        assert (d <= 20) == chases, d
        for t in (BOT_AGGRESSIVE, BOT_AGGRESSIVE_SHY):
            got = oracle_bot_decide(cfg, L, sv.blob, 0, t)
            if t == BOT_AGGRESSIVE_SHY and d < 25:
                continue  # (flees first)
            if chases:
                _expect(got, _chase_target(sv, 1, 100, loc), 1, loc)
            else:
                _expect(got, (30.0, 170.0), 0, loc)
    # within 20 but nothing edible: the nearest pellet
    for i in range(3):
        sv.cells[1][i]["mass"] = 95
    _expect(oracle_bot_decide(cfg, L, sv.blob, 0, BOT_AGGRESSIVE), (30.0, 170.0), 0, loc)
    # a largest cell of 25 eats nothing
    sv.cells[1][0]["mass"] = 10
    sv.cells[0][1]["mass"] = 25
    sv.cells[0][0]["mass"] = 25
    loc = _loc(sv, 0)
    _expect(oracle_bot_decide(cfg, L, sv.blob, 0, BOT_AGGRESSIVE), (30.0, 170.0), 0, loc)


def test_no_pellets_is_status_2_and_flags_nothing():
    cfg, L, sv = _state(bots=1)
    _cell(sv, 0, 0, 100.0, 100.0, 100)
    _cell(sv, 1, 0, 190.0, 190.0, 50)
    sv.players["action"][0] = 2
    _pellets(sv, [])
    loc = _loc(sv, 0)
    before = sv.blob.copy()
    for t in TYPES:
        dxdy, target, act, status = oracle_bot_decide(cfg, L, sv.blob, 0, t)
        assert status == BOT_NO_PELLET and act == 0 and not dxdy.any() and tuple(target) == loc
    assert np.array_equal(sv.blob, before)
    # flee and chase still decide without pellets
    _cell(sv, 1, 0, 110.0, 100.0, 50)
    _expect(oracle_bot_decide(cfg, L, sv.blob, 0, BOT_HUNGRY_SHY), (F(90), F(100)), 0, loc)
    _expect(oracle_bot_decide(cfg, L, sv.blob, 0, BOT_AGGRESSIVE), _chase_target(sv, 1, 100, loc), 2, loc)
    assert int(sv.hdr["flags"]) == 0


def test_dead_agent_and_other_types():
    cfg, L, sv = _state(A=2, bots=1)
    _cell(sv, 0, 0, 100.0, 100.0, 100)
    _cell(sv, 2, 0, 105.0, 100.0, 50)
    _pellets(sv, [(20.0, 20.0)])
    sv.players["action"][1] = 2
    for t in TYPES:
        dxdy, target, act, status = oracle_bot_decide(cfg, L, sv.blob, 1, t)
        assert status == BOT_DEAD and act == 0 and not dxdy.any() and not target.any()
    _pellets(sv, [])
    assert oracle_bot_decide(cfg, L, sv.blob, 1, BOT_HUNGRY)[3] == BOT_DEAD  # (before NO_PELLET)
    assert oracle_bot_decide(cfg, L, sv.blob, 0, -1)[3] == BOT_SKIPPED
    for t in (4, -2, 1 << 30):
        assert oracle_bot_decide(cfg, L, sv.blob, 0, t)[3] == BOT_BAD_TYPE


def test_dead_and_absent_players_are_never_chosen():
    """a mixed-task layout with an instance of mode 1 (the mode-7 bot absent), and a dead bot of a plain layout: stale cells next
    to the agent count for nothing"""
    from agarcl_b200 import _lib
    cfg = make_cfg(mode_number=1, num_bots=0, task_modes=task_bits([1, 7]), arena_size=200, num_pellets=100, num_viruses=0)
    L = _lib.make_layout(cfg)
    assert L.P == 2
    layouts = [(cfg, L)]
    cfg2, L2, _ = _state(bots=2)
    layouts.append((cfg2, L2))
    for cfg, L in layouts:
        sv = StateView(L)
        _cell(sv, 0, 0, 100.0, 100.0, 200)
        sv.players["action"][0] = 1
        _pellets(sv, [(40.0, 40.0), (180.0, 30.0)])
        clean = sv.blob.copy()
        for p in range(1, L.P):
            for i in range(4):
                _cell(sv, p, i, 101.0 + i, 100.0, 30)
            sv.players["n_cells"][p] = 0
        for t in TYPES:
            got, ref = oracle_bot_decide(cfg, L, sv.blob, 0, t), oracle_bot_decide(cfg, L, clean, 0, t)
            _expect(got, (40.0, 40.0), 0, _loc(sv, 0))
            assert all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(got, ref))


def test_the_blob_is_never_modified():
    """aged multi-agent states, every agent and type, with and without pellets"""
    for seed in (1, 2):
        o = aged_oracle(dict(num_agents=4, num_bots=8, arena_size=300, num_pellets=300, num_viruses=4), seed, 30)
        before = o.state.blob.copy()
        statuses = set()
        for a in range(o.L.A):
            for t in TYPES:
                statuses.add(oracle_bot_decide(o.cfg, o.L, o.state.blob, a, t)[3])
        n_pellets = int(o.state.hdr["n_pellets"])
        o.state.hdr["n_pellets"] = 0
        before0 = o.state.blob.copy()
        for a in range(o.L.A):
            for t in TYPES:
                statuses.add(oracle_bot_decide(o.cfg, o.L, o.state.blob, a, t)[3])
        assert np.array_equal(o.state.blob, before0)
        o.state.hdr["n_pellets"] = n_pellets
        assert np.array_equal(o.state.blob, before)
        assert BOT_DECIDED in statuses and BOT_NO_PELLET in statuses


def test_k_bot_actions_has_no_spills():
    from agarcl_b200 import build
    flags = [f for f in build.NVCC_FLAGS if f != "-shared"]
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([nvcc] + flags + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, "bot_kernel.cu"),
                                             "-o", os.path.join(d, "bot_kernel.o")], capture_output=True, text=True, check=True)
    text = r.stdout + r.stderr
    blocks = re.findall(r"Function properties for (\S*k_bot_actions\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                        r"(\d+) bytes spill loads", text)
    assert len(blocks) == 1, text
    for name, stack, st, ld in blocks:
        assert (int(stack), int(st), int(ld)) == (0, 0, 0), (name, stack, st, ld)
