#!/usr/bin/env python
"""What a mixed-task batch saves: the ten AgarCL mini-games (bench/tasks_configs, modes 1..10: arena 350, 500 pellets, no viruses,
one bot in modes 7..10, episodes of 500 / 3000 / 10000 steps) stepped with auto-reset in three arrangements:

  mixed       ONE batch of --instances instances, instance i on mode 1 + i % 10 with its mode's episode length
  ten_small   ten homogeneous batches of --instances / 10 instances (409 / 410), stepped back to back on one stream
  big_<k>     each homogeneous batch of --instances instances of mode k alone (what one mini-game costs at full occupancy)

    python tools/exp_tasks.py [--instances 4096] [--age 300] [--calls 50] [--repeats 5] [--out FILE]

Every batch is aged by --age random-walk steps first (an early step is cheaper than a steady-state one).  Each repeat times
--calls env-steps of every arm with device events around the whole arm; the arms alternate within a repeat and their order rotates
between repeats.  One JSON line per arm: ms per env-step (median / min / max over the repeats) and env-steps/s, plus the GPU's
name and power limit read in the same run."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from exp_common import RandomWalk, gpu_info, stats, time_arms, write_lines  # noqa: E402
from run_tasks_configs import TASKS  # noqa: E402

MODES = list(range(1, 11))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instances", type=int, default=4096)
    ap.add_argument("--age", type=int, default=300)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("exp_tasks.py measures on a GPU; none is visible")
    from agarcl_b200 import make_cfg
    from agarcl_b200._abi import task_bits
    from agarcl_b200.batch import Batch
    N = a.instances
    common = dict(ticks_per_step=4, num_frames=1, arena_size=350, num_pellets=500, num_viruses=0, num_bots=0, pellet_regen=True,
                  grid_size=128, reward_type=1, c_death=0)
    walk = RandomWalk(N)

    def make(n, mode, base, tasks=False):
        b = Batch(make_cfg(n_instances=n, mode_number=mode, instance_base=base, task_modes=task_bits(MODES) if tasks else 0, **common))
        b.seed(7)
        b.set_autoreset(TASKS[mode]["number_steps"])
        if tasks:
            m = torch.tensor([MODES[i % 10] for i in range(n)], dtype=torch.int32, device="cuda")
            lim = torch.tensor([TASKS[int(k)]["number_steps"] for k in m.tolist()], dtype=torch.int32, device="cuda")
            assert bool((b.set_tasks(m, lim) == 1).all())
        b.reset()
        return b

    def step(batches):  # one env-step of every batch of the arm, the actions of instance j from slot j of the shared tensors
        off = 0
        for b in batches:
            b.set_actions_device(walk.dxdy[off:].data_ptr(), walk.act[off:].data_ptr())
            b.step_autoreset()
            off += b.N

    sizes = [N // 10 + (1 if k < N % 10 else 0) for k in range(10)]
    bases = [sum(sizes[:k]) for k in range(10)]
    arms = {"mixed": [make(N, 1, 0, tasks=True)], "ten_small": [make(sizes[k], MODES[k], bases[k]) for k in range(10)]}
    for k in MODES:
        arms[f"big_{k}"] = [make(N, k, 0)]
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
                          env_steps_per_s=envs / s["median"] * 1e3, age=a.age, calls=a.calls, repeats=a.repeats, state_flags=flags[n],
                          **info))
    lines.append(dict(arm="summary", mixed_over_ten_small=lines[0]["ms_per_env_step"] / lines[1]["ms_per_env_step"], **info))
    write_lines(lines, a.out)


if __name__ == "__main__":
    main()
