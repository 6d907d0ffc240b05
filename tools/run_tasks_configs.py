#!/usr/bin/env python
"""Runs the reference's ten mini-game task configurations (bench/tasks_configs/mode_{1..10}.json: arena 350, 500 pellets, no
viruses, mode k, 0 bots (modes 1-6) or one bot of type k-7 (modes 7-10), episodes of 500 / 3000 / 10000 steps) through the
batched vector environment (agarcl_b200.gym_env.BatchedAgarioEnv: N lockstep instances, auto-reset) with the random-walk policy of
bench/go_bigger_example.py:100-103, and prints one JSON line per mode: env-steps/s, episodes finished, mean return, state flags.

    python tools/run_tasks_configs.py [--envs 4096] [--steps 600] [--modes 1 2 ...] [--dir DIR] [--mixed] [--policy POLICY]

--policy hungry | hungry_shy | aggressive | aggressive_shy drives every agent with that built-in bot instead of the random walk
(BatchedAgarioEnv.bot_actions: the reference's bot code run for the agent on the device every step, its actions fed straight into
step()), in both the per-mode and the --mixed runs: a scripted-baseline table for the mini-games.  Its JSON lines carry "policy";
the default, random, prints them as before.

--mixed runs the selected mini-games in ONE mixed-task batch of --envs instances instead of one batch per mode: instance i plays
mode modes[i % len(modes)] with that mode's episode length, every auto-reset keeps it on its mode, and the finished episodes and
returns are summed per task on the device (index_add_ on info["task"]).  It prints one JSON line per mode and one for the batch.

With --dir the mode_k.json files themselves are loaded (keys the batched grid environment does not have -- screen_len, video_path,
agent_view, render_mode, load_env_snapshot -- are ignored; obs_type "screen" is OpenGL and out of scope: the grid observation with
all channels is produced instead).  Without it the table below (the same numbers) is used, so the runner works on the GPU box."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from agarcl_b200._abi import BOT_TYPES  # noqa: E402

# bench/tasks_configs/mode_k.json, the keys that reach the engine
TASKS = {k: dict(ticks_per_step=4, num_frames=1, arena_size=350, num_pellets=500, num_viruses=0, num_bots=(1 if k >= 7 else 0),
                 pellet_regen=True, grid_size=128, reward_type=1, c_death=0, mode=k,
                 number_steps=(500 if k <= 2 else 3000 if k <= 6 else 10000), env_type=0) for k in range(1, 11)}
KEEP = set(TASKS[1])


def load_dir(d):
    out = {}
    for k in range(1, 11):
        with open(os.path.join(d, f"mode_{k}.json")) as f:
            out[k] = {key: v for key, v in json.load(f).items() if key in KEEP}
    return out


def policy_actions(args, env, gen, N, bot):
    """(dxdy, act, bot buffers) of this step: the random walk of bench/go_bigger_example.py:100-103, or the built-in bot computed
    on the device into the buffers of the previous step"""
    import torch
    if args.policy == "random":
        dxdy = (torch.rand((N, 2), device="cuda", generator=gen) * 2 - 1).float()
        act = torch.randint(0, 3, (N,), device="cuda", generator=gen, dtype=torch.int32)
        return dxdy, act, None
    bot = env.bot_actions(BOT_TYPES[args.policy], out=bot)
    return bot[0], bot[1], bot


def with_policy(args, line):
    return line if args.policy == "random" else dict(line, policy=args.policy)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--modes", type=int, nargs="*", default=list(range(1, 11)))
    ap.add_argument("--dir", default=None)
    ap.add_argument("--mixed", action="store_true")
    ap.add_argument("--policy", default="random", choices=["random"] + list(BOT_TYPES))
    args = ap.parse_args()
    import torch
    from agarcl_b200.gym_env import BatchedAgarioEnv
    tasks = load_dir(args.dir) if args.dir else TASKS
    N = args.envs
    if args.mixed:
        return run_mixed(args, tasks)
    for k in args.modes:
        kw = dict(tasks[k], observe_cells=True, observe_others=True, observe_viruses=True, observe_pellets=True)
        env = BatchedAgarioEnv(N, obs_type="grid", **kw)
        env.seed(1000 * k)
        env.reset()
        gen = torch.Generator(device="cuda")
        gen.manual_seed(k)
        # finished episodes and their returns come from info, summed on the device: the loop never waits for it
        finished = torch.zeros((), dtype=torch.int64, device="cuda")
        ret_sum = torch.zeros((), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bot = None
        for t in range(args.steps):
            dxdy, act, bot = policy_actions(args, env, gen, N, bot)
            _, _, _, _, info = env.step(dxdy, act)
            m = info["reset_mask"]
            finished += m.sum()
            ret_sum += torch.where(m, info["episode_return"], 0.0).sum()
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        finished, ret_sum = int(finished), float(ret_sum)
        f, names = env.flags()
        print(json.dumps(with_policy(args, {"task": f"mode_{k}", "envs": N, "steps": args.steps, "env_steps_per_s": N * args.steps / sec,
                                            "episode_steps": kw["number_steps"], "episodes_finished": finished,
                                            "mean_return": (ret_sum / finished) if finished else None, "state_flags": names})))
        env.close()


def run_mixed(args, tasks):
    import torch
    from agarcl_b200.gym_env import BatchedAgarioEnv
    N, modes = args.envs, list(args.modes)
    first = tasks[modes[0]]
    for k in modes:  # one batch holds the mini-games that differ in their mode only
        diff = {key for key in KEEP - {"mode", "number_steps", "num_bots"} if tasks[k][key] != first[key]}
        if diff:
            sys.exit(f"mode_{k} differs from mode_{modes[0]} in {sorted(diff)}: it cannot share a mixed-task batch")
    kw = dict(first, observe_cells=True, observe_others=True, observe_viruses=True, observe_pellets=True, num_bots=0)
    kw.pop("mode")
    env = BatchedAgarioEnv(N, obs_type="grid", tasks=modes, mode=modes[0], **kw)
    env.seed(1000)
    mode_of = torch.tensor([modes[i % len(modes)] for i in range(N)], dtype=torch.int32, device="cuda")
    limit_of = torch.tensor([tasks[int(m)]["number_steps"] for m in mode_of.tolist()], dtype=torch.int32, device="cuda")
    res = env.set_tasks(mode_of, limit_of)  # (taken by the reset below)
    env.reset()
    assert bool((res == 1).all()), "a task was rejected"
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1)
    finished = torch.zeros(11, dtype=torch.int64, device="cuda")
    ret_sum = torch.zeros(11, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bot = None
    for t in range(args.steps):
        dxdy, act, bot = policy_actions(args, env, gen, N, bot)
        _, _, _, _, info = env.step(dxdy, act)
        m = info["reset_mask"]
        task = info["task"].long()  # (after an auto-reset: the new episode's, which is the finished one's here)
        finished.index_add_(0, task, m.long())
        ret_sum.index_add_(0, task, torch.where(m, info["episode_return"], 0.0))
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    finished, ret_sum = finished.tolist(), ret_sum.tolist()
    f, names = env.flags()
    for k in modes:
        print(json.dumps(with_policy(args, {"task": f"mode_{k}", "mixed": True, "envs": sum(1 for i in range(N) if modes[i % len(modes)] == k),
                                            "steps": args.steps, "episode_steps": tasks[k]["number_steps"], "episodes_finished": finished[k],
                                            "mean_return": (ret_sum[k] / finished[k]) if finished[k] else None})))
    print(json.dumps(with_policy(args, {"task": "mixed", "modes": modes, "envs": N, "steps": args.steps, "env_steps_per_s": N * args.steps / sec,
                                        "ms_per_step": 1e3 * sec / args.steps, "state_flags": names})))
    env.close()


if __name__ == "__main__":
    main()
