#!/usr/bin/env python
"""What per-instance game sizes cost and save: --instances mode-0 instances of BASELINE.json configs[1] (1 agent, up to 25 bots,
1000 pellets, 25 viruses, arena 1000) stepped with auto-reset in four arrangements:

  plain        no task_modes (the batch as bench.py runs it)
  tasks_max    task_modes = {0}, every size at its maximum (what a mixed batch that never sets sizes costs)
  spread       task_modes = {0}, instance i on setting i % 8 of SETTINGS: bots 0 and 13..25, pellets 250..1000, viruses 0..25
  per_size     the same eight settings as eight single-size batches of --instances / 8, stepped back to back on one stream

    python tools/exp_task_sizes.py [--instances 4096] [--age 300] [--limit 500] [--calls 50] [--repeats 5] [--out FILE]

Every batch is aged by --age random-walk steps first, with auto-reset at --limit steps.  Each repeat times --calls env-steps of
every arm with device events around the whole arm; the arms alternate within a repeat and their order rotates between repeats.
One JSON line per arm: ms per env-step (median / min / max over the repeats) and env-steps/s, plus the GPU's name and power limit
read in the same run."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from exp_common import RandomWalk, gpu_info, stats, time_arms, write_lines  # noqa: E402

# (bots, pellets, viruses); bot counts 1..12 of 1 agent + 25 bots fail the player-order check (include/agarcl_b200.h)
SETTINGS = [(0, 250, 0), (13, 357, 4), (15, 464, 7), (17, 571, 11), (19, 679, 14), (21, 786, 18), (23, 893, 22), (25, 1000, 25)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instances", type=int, default=4096)
    ap.add_argument("--age", type=int, default=300)
    ap.add_argument("--limit", type=int, default=500)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("exp_task_sizes.py measures on a GPU; none is visible")
    from agarcl_b200 import make_cfg
    from agarcl_b200._abi import task_bits
    from agarcl_b200.batch import Batch
    N = a.instances
    configs1 = dict(num_agents=1, ticks_per_step=4, arena_size=1000, pellet_regen=True, num_pellets=1000, num_viruses=25, num_bots=25,
                    reward_type=1, c_death=0, mode_number=0, num_frames=1, grid_size=128)
    cap_v = configs1["num_viruses"] + 32
    walk = RandomWalk(N)

    def make(n, base, tasks=False, spread=False, size=None):
        kw = dict(configs1)
        if size is not None:
            kw.update(num_bots=size[0], num_pellets=size[1], num_viruses=size[2], cap_viruses=cap_v)
        b = Batch(make_cfg(n_instances=n, instance_base=base, task_modes=task_bits([0]) if tasks else 0, **kw))
        b.seed(7)
        b.set_autoreset(a.limit)
        if spread:
            col = [torch.tensor([SETTINGS[i % 8][k] for i in range(n)], dtype=torch.int32, device="cuda") for k in range(3)]
            assert bool((b.set_task_sizes(*col) == 1).all())
        b.reset()
        return b

    def step(batches):  # one env-step of every batch of the arm, the actions of instance j from slot j of the shared tensors
        off = 0
        for b in batches:
            b.set_actions_device(walk.dxdy[off:].data_ptr(), walk.act[off:].data_ptr())
            b.step_autoreset()
            off += b.N

    sizes = [N // 8 + (1 if k < N % 8 else 0) for k in range(8)]
    bases = [sum(sizes[:k]) for k in range(8)]
    arms = {"plain": [make(N, 0)], "tasks_max": [make(N, 0, tasks=True)], "spread": [make(N, 0, tasks=True, spread=True)],
            "per_size": [make(sizes[k], bases[k], size=SETTINGS[k]) for k in range(8)]}
    for _ in range(a.age):
        walk.next()
        for bs in arms.values():
            step(bs)
    ms = time_arms({n: (lambda bs=bs: step(bs)) for n, bs in arms.items()}, a.calls, a.repeats)
    info = gpu_info()
    flags = {n: sorted(set().union(*[set(b.flags()[1]) for b in bs])) for n, bs in arms.items()}
    lines = []
    for n, t in ms.items():
        s = stats(t)
        envs = sum(b.N for b in arms[n])
        lines.append(dict(arm=n, instances=envs, ms_per_env_step=s["median"], ms_min=s["min"], ms_max=s["max"],
                          env_steps_per_s=envs / s["median"] * 1e3, age=a.age, limit=a.limit, calls=a.calls, repeats=a.repeats,
                          state_flags=flags[n], **info))
    med = {r["arm"]: r["ms_per_env_step"] for r in lines}
    lines.append(dict(arm="summary", tasks_max_over_plain=med["tasks_max"] / med["plain"], spread_over_per_size=med["spread"] / med["per_size"],
                      **info))
    write_lines(lines, a.out)


if __name__ == "__main__":
    main()
