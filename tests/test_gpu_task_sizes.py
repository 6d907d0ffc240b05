"""Game sizes per instance in mixed-task batches (agarcl_batch_set_task_sizes, include/agarcl_b200.h): an instance with current
(mode, bots, pellets, viruses) steps bit for bit like the same instance of a batch created with those counts; new sizes start at
the instance's next reset and not before; bad sizes are rejected per instance on the device; snapshots, start states and JSON
carry the sizes; nothing makes the host wait."""
import json

import numpy as np
import pytest

from agarcl_b200 import make_cfg
from agarcl_b200._abi import task_bits
from agarcl_b200._lib import make_layout
from gpu_parity_lib import assert_no_host_wait, i32
from test_gpu_tasks import assert_same_game

SEEDS_BASE, BASE = 700, 40
# a crowded mode-0 arena: bots eat the agents, so mode 0 respawns players next to the absent ones
CROWDED = dict(arena_size=220, num_pellets=400, num_viruses=10, num_bots=12, grid_size=32)
# (bots, pellets, viruses): b = 0 and b = max, no pellets, no viruses, and the maxima
SETTINGS = [(0, 400, 10), (12, 400, 10), (12, 0, 0), (5, 200, 3), (1, 50, 10), (12, 100, 1), (7, 400, 0), (3, 300, 5)]


def _batch(N, **kw):
    from agarcl_b200.batch import Batch
    b = Batch(make_cfg(n_instances=N, instance_base=BASE, **kw))
    b.seed(np.arange(N, dtype=np.uint64) + SEEDS_BASE)
    return b


def _actions(rng, n):
    return rng.uniform(-1, 1, size=(n, 2)).astype(np.float32), rng.integers(0, 3, size=n).astype(np.int32)


def _pics(b, what):
    if what == "pixels":
        return b.pixels().cpu().numpy()
    return b.obs_tensor().cpu().numpy()


def _identity(N, base, modes, task_of, path, steps, min_absent_respawns=0):
    """a mixed batch of `modes` (instance i plays task_of(i) = (mode, bots, pellets, viruses)) against one batch per distinct task,
    created with those counts and the mixed batch's cap_viruses, every step for `steps` random steps"""
    import torch
    kw = dict(base, mode_number=modes[0])
    if path == "ram":
        kw["ram_obs"] = 1
    if path == "pixels":
        kw["pixel_obs"] = 32
    cap_v = base["num_viruses"] + 32
    mixed = _batch(N, task_modes=task_bits(modes), **kw)
    tasks = [task_of(i) for i in range(N)]
    assert (mixed.set_tasks(i32([t[0] for t in tasks])).cpu().numpy() == 1).all()
    res = mixed.set_task_sizes(i32([t[1] for t in tasks]), i32([t[2] for t in tasks]), i32([t[3] for t in tasks]))
    assert (res.cpu().numpy() == 1).all()
    alone = {t: _batch(N, **dict(kw, mode_number=t[0], num_bots=t[1], num_pellets=t[2], num_viruses=t[3], cap_viruses=cap_v))
             for t in set(tasks)}
    for b in [mixed] + list(alone.values()):
        b.reset()
    sz = {k: v.cpu().numpy() for k, v in mixed.task_sizes().items()}
    assert sz["bots"].tolist() == [t[1] for t in tasks] and sz["pellets"].tolist() == [t[2] for t in tasks]
    assert sz["viruses"].tolist() == [t[3] for t in tasks]
    rng = np.random.default_rng(11)
    A = mixed.A
    absent_respawns = 0
    for t in range(steps + 1):
        if t:
            acts = _actions(rng, N * A)
            for b in [mixed] + list(alone.values()):
                b.set_actions(*acts)
                b.step()
        torch.cuda.synchronize()
        mo, mr, md = _pics(mixed, path), mixed.rewards_tensor().cpu().numpy(), mixed.dones_tensor().cpu().numpy()
        ram = mixed.ram_tensor().cpu().numpy() if path == "ram" else None
        al = {k: (_pics(b, path), b.rewards_tensor().cpu().numpy(), b.dones_tensor().cpu().numpy()) for k, b in alone.items()}
        full = t % 25 == 0 or t == steps
        for i in range(N):
            k = tasks[i]
            s = slice(i * A, (i + 1) * A)
            assert np.array_equal(mo[s], al[k][0][s]), f"step {t}: observation of instance {i} {k}"
            assert np.array_equal(mr[s], al[k][1][s]) and np.array_equal(md[s], al[k][2][s]), f"step {t}: reward / done of {i} {k}"
            if ram is not None:
                assert np.array_equal(ram[i, :alone[k].layout.P], alone[k].ram_tensor().cpu().numpy()[i]), f"step {t}: ram of {i}"
            if full or (k[0] == 0 and k[1] < base["num_bots"]):
                st = mixed.download_state(i)
                if k[0] == 0 and k[1] < base["num_bots"] and t:
                    lo = int(st.hdr["respawned_lo"]) | int(st.hdr["respawned_hi"]) << 32
                    absent_respawns += lo != 0
                    assert lo >> (A + k[1]) == 0, f"step {t}: an absent player of {i} was respawned"
                if full:
                    assert_same_game(st, alone[k].download_state(i), f"step {t}: instance {i} {k}")
    assert absent_respawns >= min_absent_respawns, "no mode-0 respawn happened beside absent players"
    want = 0
    for b in alone.values():
        want |= b.flags()[0]
    assert mixed.flags()[0] == want  # (bots may reach a libc rand() site in the crowded arena: RAND_SITE, in both alike)
    for b in [mixed] + list(alone.values()):
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["grid", "ram", "pixels"])
def test_mode0_sizes_equal_single_size_batches(path):
    """N = 16 mode-0 instances with sizes spread over the range (b = 0 and b = max included) against one batch per size"""
    _identity(16, CROWDED, [0], lambda i: (0,) + SETTINGS[i % len(SETTINGS)], path, 300, min_absent_respawns=5)


@pytest.mark.gpu
@pytest.mark.parametrize("modes, bots", [((0, 7, 8), 1), ((0, 1, 3, 4), 0)])
def test_mixed_modes_with_sizes_equal_single_size_batches(modes, bots):
    """mode 0 beside modes of its bot count (the only sets a mixed batch with mode 0 accepts), each instance with its own pellets
    and viruses, and in the first set bots 0 or 1 in mode 0"""
    base = dict(arena_size=350, num_pellets=500, num_viruses=6, num_bots=bots, grid_size=48)

    def task_of(i):
        m = modes[i % len(modes)]
        return (m, (i // len(modes)) % (bots + 1) if m == 0 else bots, (120, 500, 0, 333)[i % 4], (0, 6, 2)[i % 3])
    _identity(20, base, list(modes), task_of, "grid", 200)


def _small(N=8, **kw):
    b = _batch(N, mode_number=0, task_modes=task_bits([0]), **dict(CROWDED, **kw))
    return b


@pytest.mark.gpu
def test_new_sizes_start_at_the_next_reset():
    """set_task_sizes changes nothing until the instance's next reset -- host reset, device reset and auto-reset alike; instances
    that are not reset stay bit-identical to a twin without the call"""
    import torch
    N = 8
    a, twin = _small(N), _small(N)
    rng = np.random.default_rng(5)

    def step(k, auto=False):
        for _ in range(k):
            acts = _actions(rng, N)
            for b in (a, twin):
                b.set_actions(*acts)
                b.step_autoreset() if auto else b.step()
        torch.cuda.synchronize()

    def same(instances):
        for i in instances:
            assert np.array_equal(a.download_state(i).blob, twin.download_state(i).blob), i

    for b in (a, twin):
        b.reset()
    step(5)
    new = [(2, 100, 1), (0, 400, 10), (12, 0, 0), (6, 250, 4)]
    sel = [1, 3, 4, 6]
    bots, pel, vir = ([-1] * N for _ in range(3))
    for i, (nb, npl, nv) in zip(sel, new):
        bots[i], pel[i], vir[i] = nb, npl, nv
    assert a.set_task_sizes(i32(bots), i32(pel), i32(vir)).cpu().numpy().tolist() == [1 if i in sel else 0 for i in range(N)]
    sz = a.task_sizes()
    assert sz["bots"].cpu().numpy().tolist() == [12] * N
    assert sz["next_pellets"].cpu().numpy().tolist() == [pel[i] if i in sel else 400 for i in range(N)]
    step(10)
    same(range(N))
    # device reset of instances 1 and 4: they take the new sizes, the rest is untouched
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
    mask[[1, 4]] = 1
    for b in (a, twin):
        b.reset_device(mask)
    torch.cuda.synchronize()
    for i in (1, 4):
        nb, npl, nv = new[sel.index(i)]
        assert (int(sz["bots"][i]), int(sz["pellets"][i]), int(sz["viruses"][i])) == (nb, npl, nv)
        st = a.download_state(i)
        assert int(st.hdr["n_pellets"]) == npl and int(st.hdr["n_viruses"]) == nv and int(st.hdr["next_cell_id"]) == 2 + nb
        assert (st.players["n_cells"][:1 + nb] == 1).all() and (st.players["n_cells"][1 + nb:] == 0).all()
    same([i for i in range(N) if i not in (1, 4)])
    step(5)
    same([0, 2, 5, 7])
    # host reset: every instance takes its pending sizes
    for b in (a, twin):
        b.reset()
    torch.cuda.synchronize()
    assert sz["viruses"].cpu().numpy().tolist() == [vir[i] if i in sel else 10 for i in range(N)]
    same([0, 2, 5, 7])
    # auto-reset: the truncation at the limit starts the next episode with the new sizes
    assert a.set_task_sizes(None, None, i32([0] * N)).cpu().numpy().tolist() == [1] * N
    for b in (a, twin):
        b.set_autoreset(6)
    old = [vir[i] if i in sel else 10 for i in range(N)]
    reset = np.zeros(N, bool)
    for _ in range(10):
        step(1, auto=True)
        reset |= a.episode()["reset_mask"].cpu().numpy().astype(bool)
        assert sz["viruses"].cpu().numpy().tolist() == [0 if reset[i] else old[i] for i in range(N)]
    assert reset.all()
    assert sz["pellets"].cpu().numpy().tolist() == [pel[i] if i in sel else 400 for i in range(N)]
    for i in range(N):
        assert int(a.download_state(i).hdr["n_viruses"]) == 0
    a.close()
    twin.close()


def _order(P):
    return list(make_layout(make_cfg(num_agents=P, num_bots=0, mode_number=1)).order)[:P]


def _agents_with_a_refused_bot_count():
    """(A, num_bots, refused counts): the first multi-agent mode-0 batch whose player order, restricted to A + b players, is not
    the order of A + b players alone for some b"""
    for A in range(2, 40):
        for nb in range(1, 9):
            full = _order(A + nb)
            bad = [b for b in range(nb + 1) if [p for p in full if p < A + b] != _order(A + b)]
            if bad:
                return A, nb, bad
    raise AssertionError("no such batch")


@pytest.mark.gpu
def test_rejections():
    import torch
    from agarcl_b200._lib import AgarclError
    N = 6
    b = _small(N)
    b.reset()
    res = b.set_task_sizes(i32([13, 12, -2, 4, -1, -1]), i32([10, 401, 5, -1, -1, 0]), i32([0, 0, 0, 11, -1, -5]))
    torch.cuda.synchronize()
    # bots above max / pellets above max / bots -2 / viruses above max / all kept / viruses -5
    assert res.cpu().numpy().tolist() == [2, 2, 2, 2, 0, 2]
    sz = b.task_sizes()
    for k, v in (("next_bots", 12), ("next_pellets", 400), ("next_viruses", 10)):
        assert sz[k].cpu().numpy().tolist() == [v] * N, k  # a rejected instance keeps every pending size
    # NULL arrays keep every pending value; -1 keeps one entry
    assert b.set_task_sizes(None, i32([7, -1, 7, -1, 7, -1])).cpu().numpy().tolist() == [1, 0, 1, 0, 1, 0]
    assert b.set_task_sizes().cpu().numpy().tolist() == [0] * N
    assert sz["next_pellets"].cpu().numpy().tolist() == [7, 400] * 3 and sz["next_bots"].cpu().numpy().tolist() == [12] * N
    with pytest.raises(AgarclError, match="bots"):
        b.set_task_sizes(i32([1] * (N - 1)))
    b.close()
    # a bot count whose players the batch's order does not hold (several agents)
    A, nb, bad = _agents_with_a_refused_bot_count()
    m = _batch(4, mode_number=0, task_modes=task_bits([0]), num_agents=A, num_bots=nb, arena_size=300, num_pellets=50,
               num_viruses=0, grid_size=16)
    good = [x for x in range(nb + 1) if x not in bad]
    res = m.set_task_sizes(i32([bad[0], good[0], bad[-1], -1]))
    assert res.cpu().numpy().tolist() == [2, 1, 2, 0]
    assert m.task_sizes()["next_bots"].cpu().numpy().tolist() == [nb, good[0], nb, nb]
    m.close()
    # one agent: every count is allowed
    one = _small(13)
    assert (one.set_task_sizes(i32(list(range(13)))).cpu().numpy() == 1).all()
    one.close()
    plain = _batch(2, mode_number=0, **CROWDED)
    with pytest.raises(AgarclError, match="without task_modes"):
        plain.set_task_sizes(i32([1, 1]))
    with pytest.raises(AgarclError, match="without task_modes"):
        plain.task_sizes()
    plain.close()


@pytest.mark.gpu
def test_set_task_sizes_and_step_autoreset_do_not_wait_for_the_device():
    import torch
    N = 64
    b = _small(N)
    b.reset()
    b.set_autoreset(20)
    bots = i32([i % 13 for i in range(N)])
    s = torch.cuda.Stream()
    for _ in range(2):
        b.set_task_sizes(bots, stream=s.cuda_stream)
        b.step_autoreset(stream=s.cuda_stream)

    def calls():
        b.set_task_sizes(bots, None, bots, stream=s.cuda_stream)
        b.step_autoreset(stream=s.cuda_stream)

    assert_no_host_wait(calls, s)
    b.close()


@pytest.mark.gpu
def test_snapshots_start_states_and_json_carry_the_sizes(tmp_path):
    import torch
    N, j = 8, 5
    src, dst = _small(N), _small(N)
    assert (src.set_task_sizes(i32([3] * N), i32([150] * N), i32([2] * N)).cpu().numpy() == 1).all()
    rng = np.random.default_rng(9)
    for b in (src, dst):
        b.reset()

    def step(k, bs):
        for _ in range(k):
            acts = _actions(rng, N)
            for b in bs:
                b.set_actions(*acts)
                b.step()
        torch.cuda.synchronize()

    step(20, (src, dst))
    pool = src.snapshot_pool(4)
    src.save_states(pool, i32([j]))
    torch.cuda.synchronize()
    hdr = pool[0, :64].cpu().numpy().view(np.int32)
    assert hdr[9] == 0x5A534741 and hdr[10:13].tolist() == [3, 150, 2]  # sizes_marker, task_bots, task_pellets, task_viruses
    # restore at the same global index: the sizes become current and the game goes on like its source
    res = dst.restore_states(pool, i32([0 if i == j else -1 for i in range(N)]))
    assert res.cpu().numpy().tolist() == [1 if i == j else 0 for i in range(N)]
    sz = dst.task_sizes()
    assert (int(sz["bots"][j]), int(sz["pellets"][j]), int(sz["viruses"][j])) == (3, 150, 2)
    assert int(sz["next_bots"][j]) == 12  # the pending sizes are the destination's own
    for t in range(40):
        step(1, (src, dst))
        assert np.array_equal(src.download_state(j).blob, dst.download_state(j).blob), t
        assert np.array_equal(src.obs_tensor()[j].cpu().numpy(), dst.obs_tensor()[j].cpu().numpy()), t
    # a slot without the marker (saved before sizes were stored) restores with the maxima; a bot count above the maximum is refused
    pool[1] = pool[0]
    pool[1, 36:52] = 0
    pool[2] = pool[0]
    pool[2, 40:44] = torch.tensor(np.array([13], np.int32).view(np.uint8), device="cuda")
    res = dst.restore_states(pool, i32([1, 2, -1, -1, -1, -1, -1, -1]))
    assert res.cpu().numpy().tolist() == [1, 2, 0, 0, 0, 0, 0, 0]
    assert (int(sz["bots"][0]), int(sz["pellets"][0]), int(sz["viruses"][0])) == (12, 400, 10)
    assert (int(sz["bots"][1]), int(sz["pellets"][1]), int(sz["viruses"][1])) == (12, 400, 10)
    # start states: a reset of instance 2 begins in slot 0 and plays its sizes
    dst.set_start_states(pool, i32([-1, -1, 0, -1, -1, -1, -1, -1]))
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
    mask[2] = 1
    dst.reset_device(mask)
    torch.cuda.synchronize()
    assert dst.start_result().cpu().numpy()[2] == 1
    assert (int(sz["bots"][2]), int(sz["pellets"][2]), int(sz["viruses"][2])) == (3, 150, 2)
    dst.set_start_states(None)
    # JSON: the instance's current sizes travel with it
    path = tmp_path / "sizes.json"
    src.save_env_state(j, path)
    with open(path) as f:
        js = json.load(f)
    assert (js["num_bots"], js["num_pellets"], js["num_viruses"]) == (3, 150, 2) and len(js["players"]) == 4
    dst.load_env_state(6, path, lossless=True)
    assert (int(sz["bots"][6]), int(sz["pellets"][6]), int(sz["viruses"][6])) == (3, 150, 2)
    assert_same_game(dst.download_state(6), src.download_state(j), "JSON load")
    for b in (src, dst):
        b.close()


@pytest.mark.gpu
def test_sets_without_mode_0_accept_every_bot_count(tmp_path):
    """without mode 0 the bot count means nothing: a batch of modes {1, 7} with num_bots = 25 (more than its layout's players)
    keeps restoring its own slots, takes pellets-only sizes and reloads its own JSON; a JSON of a plain mode-7 batch of 25 bots
    loads into a {7, 8} batch of num_bots 1"""
    import torch
    N = 4
    kw = dict(arena_size=350, num_pellets=500, num_viruses=4, num_bots=25, grid_size=32)
    b = _batch(N, mode_number=7, task_modes=task_bits([1, 7]), **kw)
    assert b.layout.P == 2
    assert b.set_tasks(i32([1, 7, 7, 1])).cpu().numpy().tolist() == [1] * N
    assert b.set_task_sizes(None, i32([200, 300, -1, 100])).cpu().numpy().tolist() == [1, 1, 0, 1]
    assert b.set_task_sizes(i32([0, 3, 25, -1])).cpu().numpy().tolist() == [1, 1, 1, 0]
    assert b.set_task_sizes(i32([26, -1, -1, -1])).cpu().numpy().tolist() == [2, 0, 0, 0]
    b.reset()
    sz = b.task_sizes()
    assert sz["pellets"].cpu().numpy().tolist() == [200, 300, 500, 100] and sz["bots"].cpu().numpy().tolist() == [0, 3, 25, 25]
    assert int(b.download_state(1).hdr["n_pellets"]) == 300 and int(b.download_state(2).hdr["n_pellets"]) == 500
    rng = np.random.default_rng(3)
    for _ in range(10):
        b.set_actions(*_actions(rng, N))
        b.step()
    pool = b.snapshot_pool(N)
    b.save_states(pool, i32(list(range(N))))
    assert b.restore_states(pool, i32([3, 2, 1, 0])).cpu().numpy().tolist() == [1] * N
    assert sz["bots"].cpu().numpy().tolist() == [25, 25, 3, 0]
    marker_less = pool.clone()
    marker_less[:, 36:52] = 0
    assert b.restore_states(marker_less, i32([0, -1, -1, -1])).cpu().numpy().tolist() == [1, 0, 0, 0]
    assert (int(sz["bots"][0]), int(sz["pellets"][0]), int(sz["viruses"][0])) == (25, 500, 4)
    b.set_start_states(pool, i32([1, 1, -1, -1]))
    mask = torch.tensor([1, 1, 0, 0], dtype=torch.uint8, device="cuda")
    b.reset_device(mask)
    torch.cuda.synchronize()
    assert b.start_result().cpu().numpy().tolist()[:2] == [1, 1]
    assert sz["pellets"].cpu().numpy().tolist()[:2] == [300, 300]
    b.set_start_states(None)
    path = tmp_path / "own.json"
    b.save_env_state(1, path)
    b.load_env_state(2, path, lossless=True)
    assert_same_game(b.download_state(2), b.download_state(1), "JSON round trip")
    assert (int(sz["bots"][2]), int(sz["pellets"][2])) == (25, 300)
    b.close()
    plain7 = _batch(2, mode_number=7, **kw)
    plain7.reset()
    path7 = tmp_path / "plain7.json"
    plain7.save_env_state(0, path7)
    m78 = _batch(2, mode_number=7, task_modes=task_bits([7, 8]), **dict(kw, num_bots=1))
    m78.reset()
    m78.load_env_state(1, path7, lossless=True)
    assert_same_game(m78.download_state(1), plain7.download_state(0), "JSON of a plain mode-7 batch")
    assert int(m78.task_sizes()["bots"][1]) == 1
    for x in (plain7, m78):
        x.close()
