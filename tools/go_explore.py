#!/usr/bin/env python
"""Go-Explore on one mini-game with the device archive (BatchedAgarioEnv.set_archive): the exploration phase is step() in a
loop -- every step files each game under its cell and keeps the best game per cell, every finished episode returns to a cell
drawn with weight 1 / (1 + isqrt(times chosen)).  The same number of env-steps without returns (an archive with select = 0:
it counts cells, every episode spawns afresh) is the baseline.

    python tools/go_explore.py [--mode 1] [--envs 1024] [--steps 2000] [--episode 100] [--cells 16] [--slots 16384]
                               [--policy random|hungry] [--every 250] [--out FILE]

Every agent explores with a random walk (a new direction every step; split and feed with probability 1/8 each) or with the
built-in Hungry bot (--policy hungry).  Prints one JSON line per checkpoint and arm: env-steps so far, cells found (entries in
use plus those dropped from a full archive), the best trajectory score of any cell and the longest trajectory kept."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def run(a, select):
    import torch
    from agarcl_b200 import BOT_HUNGRY
    from agarcl_b200.gym_env import BatchedAgarioEnv
    env = BatchedAgarioEnv(a.envs, mode=a.mode, number_steps=a.episode)
    env.seed(a.seed)
    env.reset()
    env.set_archive(a.slots, cells_per_side=a.cells, select=select, seed=a.seed)
    g = torch.Generator(device="cuda").manual_seed(a.seed)
    NA = a.envs * env.num_agents
    dxdy, act = torch.empty((NA, 2), device="cuda"), torch.empty(NA, dtype=torch.int32, device="cuda")
    out = []
    for t in range(1, a.steps + 1):
        if a.policy == "hungry":
            dxdy, act, _ = env.bot_actions(BOT_HUNGRY)
        else:
            dxdy.uniform_(-1, 1, generator=g)
            r = torch.rand(NA, device="cuda", generator=g)
            act = ((r < 0.125).int() * 1 + (r > 0.875).int() * 2).int()
        env.step(dxdy, act)
        if t % a.every == 0 or t == a.steps:
            ar = {k: v.cpu().numpy() for k, v in env.archive().items()}
            used, dropped, improved = (int(x) for x in ar["counters"])
            out.append(dict(arm="go_explore" if select else "no_returns", mode=a.mode, policy=a.policy, envs=a.envs, step=t,
                            env_steps=t * a.envs, cells_found=used + dropped, entries=used, improved=improved,
                            best_score=float(ar["entry_score"][:used].max()) if used else None,
                            longest_trajectory=int(ar["entry_length"][:used].max()) if used else None))
    env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", type=int, default=1)
    ap.add_argument("--envs", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--episode", type=int, default=100)
    ap.add_argument("--cells", type=int, default=16)
    ap.add_argument("--slots", type=int, default=16384)
    ap.add_argument("--policy", choices=("random", "hungry"), default="random")
    ap.add_argument("--every", type=int, default=250)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("go_explore.py runs on a GPU; none is visible")
    lines = run(a, True) + run(a, False)
    text = "\n".join(json.dumps(x) for x in lines)
    print(text, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
