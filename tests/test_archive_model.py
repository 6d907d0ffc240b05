"""The archive model (archive_model.py) on crafted games, without a GPU: cell keys on bin borders and at the arena's edge, masses
at powers of two, a dead agent, winners under ties in score and length, a full archive, the selection weights and draws."""
import numpy as np

from agarcl_b200 import make_cfg
from agarcl_b200._abi import StateView
from agarcl_b200._lib import make_layout
from archive_model import ArchiveModel, bin_of, cell_key, draw_word, weight

W = 300


def _layout(num_agents=1):
    return make_layout(make_cfg(n_instances=1, num_agents=num_agents, num_bots=0, arena_size=W, num_pellets=10, num_viruses=0))


def _game(L, cells, agent=0):
    """a blob whose agent has the cells [(x, y, mass), ...] in that order"""
    sv = StateView(L)
    sv.players["n_cells"][agent] = len(cells)
    for k, (x, y, m) in enumerate(cells):
        sv.cells[agent][k]["x"], sv.cells[agent][k]["y"], sv.cells[agent][k]["mass"] = x, y, m
    return sv


def test_bins_on_borders_and_at_the_edge():
    n = 8  # bins of 37.5 units
    assert bin_of(np.float32(0.0), n, W) == 0
    assert bin_of(np.float32(37.5), n, W) == 1  # exactly on a border: the upper bin
    assert bin_of(np.nextafter(np.float32(37.5), np.float32(0)), n, W) == 0
    assert bin_of(np.float32(W), n, W) == n - 1  # x = W is clamped into the last bin
    assert bin_of(np.float32(-3.0), n, W) == 0
    assert bin_of(np.float32(1e30), n, W) == n - 1
    L = _layout()
    assert cell_key(_game(L, [(75.0, 150.0, 10)]), 0, n, W) == (3 * n + 4) * n + 2
    # the centroid is the fp32 one: (10 * 37 + 30 * 38) / 40 = 37.75 -> bin 1 at n = 8
    assert cell_key(_game(L, [(37.0, 0.0, 10), (38.0, 0.0, 30)]), 0, n, W) == (5 * n + 0) * n + 1
    assert cell_key(_game(L, [(W, W, 1)]), 0, 1, W) == 0


def test_masses_at_powers_of_two_and_a_dead_agent():
    L = _layout()
    n = 4
    for m, mb in ((1, 0), (2, 1), (3, 1), (4, 2), (1023, 9), (1024, 10), (1 << 31, 31), (0xFFFFFFFF, 31)):
        assert cell_key(_game(L, [(1.0, 1.0, m)]), 0, n, W) == mb * n * n, m
    assert cell_key(_game(L, [(1.0, 1.0, 512), (2.0, 2.0, 512)]), 0, n, W) == 10 * n * n  # the total mass counts
    assert cell_key(_game(L, []), 0, n, W) == -1
    two = _layout(num_agents=2)
    sv = _game(two, [(200.0, 10.0, 20)], agent=1)
    assert cell_key(sv, 0, n, W) == -1 and cell_key(sv, 1, n, W) == (4 * n + 0) * n + 2


def _update(model, games, rewards, dones=None, ret=None, steps=None):
    N, A = len(games), model.A
    return model.update(games, np.zeros(N * A, np.uint8) if dones is None else np.asarray(dones, np.uint8),
                        np.asarray(rewards, np.float64), np.zeros(N * A) if ret is None else np.asarray(ret, np.float64),
                        np.zeros(N, np.int64) if steps is None else np.asarray(steps, np.int64))


def test_winners_ties_and_replacement():
    L = _layout()
    g = _game(L, [(10.0, 10.0, 10)])
    other = _game(L, [(290.0, 290.0, 10)])
    m = ArchiveModel(N=5, A=1, K=4, n=4, agent=0, W=W)
    # instance 3 has the highest score; instance 4 is done by the game and is no candidate
    saves = _update(m, [g, g, other, g, g], [1.0, 1.0, 0.5, 2.0, 9.0], dones=[0, 0, 0, 0, 1])
    k, k2 = cell_key(g, 0, 4, W), cell_key(other, 0, 4, W)
    assert saves == {0: 2, 1: 3}  # new entries numbered in ascending order of their winner's instance
    assert m.key_entry[k2] == 0 and m.key_entry[k] == 1 and m.visits[k] == 3 and m.visits[k2] == 1
    assert m.cell_of.tolist() == [k, k, k2, k, k]
    # equal scores: the shorter trajectory wins; equal score and length: the lower instance
    assert (m.entry_score[1], m.entry_length[1]) == (2.0, 1)
    saves = _update(m, [g, g, g, g, g], [2.0] * 5, steps=[5, 3, 3, 9, 7])  # winner: instance 1 (length 4, before 2): not shorter
    assert saves == {} and m.entry_length[1] == 1 and m.improved == 0
    m.entry_length[1] = 10
    saves = _update(m, [g, g, g, g, g], [2.0] * 5, steps=[5, 3, 3, 9, 7])
    assert saves == {1: 1} and m.entry_length[1] == 4 and m.improved == 1
    # a higher score replaces whatever the length
    saves = _update(m, [g] * 5, [0.0] * 5, ret=[0, 0, 0, 0, 5.0], steps=[0, 0, 0, 0, 400])
    assert saves == {1: 4} and m.entry_score[1] == 5.0 and m.entry_length[1] == 401 and m.improved == 2
    # the base counts: the trajectory of an episode started from a cell
    m.base_score[0], m.base_length[0] = 10.0, 3
    saves = _update(m, [g] * 5, [0.0] * 5)
    assert saves == {1: 0} and m.entry_score[1] == 10.0 and m.entry_length[1] == 4


def test_a_full_archive_drops_new_cells_and_still_counts_visits():
    L = _layout()
    games = [_game(L, [(10.0 + 75 * k, 10.0, 10)]) for k in range(4)]
    m = ArchiveModel(N=4, A=1, K=2, n=4, agent=0, W=W)
    saves = _update(m, games[::-1], [0.0] * 4)  # instance 0 holds games[3]
    assert saves == {0: 0, 1: 1} and m.used == 2 and m.dropped == 2
    assert [int(m.visits[cell_key(g, 0, 4, W)]) for g in games] == [1, 1, 1, 1]
    assert m.key_entry[cell_key(games[3], 0, 4, W)] == 0 and m.key_entry[cell_key(games[1], 0, 4, W)] == -1
    saves = _update(m, games, [1.0] * 4)
    assert saves == {1: 2, 0: 3} and m.dropped == 4 and m.improved == 2


def test_weights_and_draws():
    assert [weight(c) for c in (0, 3, 4, 10 ** 6)] == [1 << 20, (1 << 20) // 2, (1 << 20) // 3, (1 << 20) // 1001]
    assert weight(8) == (1 << 20) // 3 and weight(9) == (1 << 20) // 4
    m = ArchiveModel(N=6, A=1, K=4, n=4, agent=0, W=W, seed=(7 << 32) | 3, instance_base=100)
    assert m.select(np.ones(6, bool)) == {i: -1 for i in range(6)} and not m.draws.any()  # an empty archive: every one spawns
    m.used = 3
    m.entry_chosen[:3] = [0, 4, 10 ** 6]
    mask = np.array([1, 0, 1, 1, 0, 1], bool)
    w = [weight(c) for c in (0, 4, 10 ** 6)]
    prefix = np.cumsum(w)
    want = {}
    for i in np.flatnonzero(mask):
        x = draw_word(m.seed, 100 + int(i), 0) % int(prefix[-1])
        want[int(i)] = int(np.argmax(prefix > x))
    picks = m.select(mask)
    assert picks == want and m.draws.tolist() == [1, 0, 1, 1, 0, 1]
    assert m.entry_chosen[:3].tolist() == [sum(1 for e in want.values() if e == k) + c for k, c in enumerate((0, 4, 10 ** 6))]
    assert draw_word(m.seed, 100, 1) != draw_word(m.seed, 100, 0) != draw_word(m.seed, 101, 0)
    m.set_base(mask, {0: 1, 2: 3})  # slot 3 is not an entry in use
    assert m.base_length.tolist()[:3] == [int(m.entry_length[1]), 0, 0]
