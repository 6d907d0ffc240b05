#!/usr/bin/env python
"""What auto-reset costs per step: bare `step`, the host composition a vector environment used before auto-reset moved to the
device (step, the reset mask from torch ops on the step counter, `bool(mask.any())`, the mask copied to the host and
`agarcl_batch_reset(host mask)`), and `agarcl_batch_step_autoreset`.  Each arm steps its own batch from the same seed with the
same device actions; the arms alternate, repeat after repeat, so drifts of the shared machine fall on all three alike.

    python tools/exp_autoreset.py [--steps 80] [--warmup 20] [--repeats 5] [--profile DIR]

One JSON line per workload, window and arm: ms per step from device events (first to last step of a repeat) and from a host
clock that ends in a synchronise, median / min / max over the repeats, and the GPU's name and power limit read in the same
run.  Two windows: steps before any instance reaches the limit (all three arms, with each arm's difference to bare `step` in
the same repeat), and steps 480-560, which contain the step on which every instance reaches it (the two resetting arms).
Workloads: BASELINE.json configs[1] (4096 instances, default arena and bots, 128x128 grid) and the mode-8 mini-game of
bench/tasks_configs (arena 350, 500 pellets, one bot) at 4096 instances; both episodic with number_steps = 500."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from exp_common import gpu_info, stats  # noqa: E402

WORKLOADS = {
    "configs1": dict(n_instances=4096),
    "mode8": dict(n_instances=4096, mode_number=8, num_bots=1, arena_size=350, num_pellets=500, num_viruses=0),
}
MAX_STEPS = 500


class Arm:
    def __init__(self, name, cfg, seed):
        import torch
        from agarcl_b200.batch import Batch
        self.name, self.b = name, Batch(cfg)
        self.b.seed(seed)
        self.b.reset()
        self.N, self.A = self.b.N, self.b.A
        self.resets = 0
        if name == "step_autoreset":
            self.b.set_autoreset(MAX_STEPS)
        elif name == "host_composition":
            self.steps = torch.zeros(self.N, dtype=torch.int64, device="cuda")
            # what its reset path runs, once before any timing (the first boolean index_put loads its kernel module)
            none = torch.zeros(self.N, dtype=torch.bool, device="cuda")
            self.b.reset(none.to(torch.uint8).cpu().numpy())
            self.steps[none] = 0

    def step(self, dxdy, act, count):
        import torch
        b = self.b
        b.set_actions_device(dxdy.data_ptr(), act.data_ptr())
        if self.name == "step":
            b.step()
        elif self.name == "step_autoreset":
            b.step_autoreset()
        else:  # the pre-device BatchedAgarioEnv.step
            b.step()
            done = b.dones_tensor().view(self.N, self.A).bool() | (self.steps >= MAX_STEPS).unsqueeze(1)
            self.steps += 1
            mask = done.any(dim=1)
            if bool(mask.any()):
                b.reset(mask.to(torch.uint8).cpu().numpy())
                self.steps[mask] = 0
                if count:
                    self.resets += int(mask.sum())


def _timed(arms, acts, first, repeats, steps):
    """ms per step of every arm, repeat after repeat, arms alternating: ({arm: [event ms]}, {arm: [host ms]})"""
    import torch
    dev_ms, host_ms = {a.name: [] for a in arms}, {a.name: [] for a in arms}
    for r in range(repeats):
        base = first + r * steps
        for arm in arms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record()
            for t in range(steps):
                arm.step(*acts[(base + t) % len(acts)], True)
            e1.record()
            torch.cuda.synchronize()
            host_ms[arm.name].append((time.perf_counter() - t0) * 1e3 / steps)
            dev_ms[arm.name].append(e0.elapsed_time(e1) / steps)
    return dev_ms, host_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=80, help="steps per repeat of the window without resets")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--workloads", nargs="*", default=list(WORKLOADS))
    ap.add_argument("--profile", default=None, help="also write a torch.profiler kernel table of 20 step_autoreset calls here")
    args = ap.parse_args()
    import torch
    from agarcl_b200 import make_cfg
    assert torch.cuda.is_available(), "exp_autoreset measures on the GPU: no CUDA device"
    quiet_end = args.warmup + args.repeats * args.steps
    assert quiet_end <= MAX_STEPS - 20, "the first window must end before the step limit"
    info = gpu_info()
    for wl in args.workloads:
        cfg = make_cfg(**WORKLOADS[wl])
        arms = [Arm(n, cfg, 1000) for n in ("step", "host_composition", "step_autoreset")]
        N, A = arms[0].N, arms[0].A
        g = torch.Generator(device="cuda")
        g.manual_seed(5)
        # the same actions for every arm, generated before any timing
        acts = [((torch.rand((N * A, 2), device="cuda", generator=g) * 2 - 1).contiguous(),
                 torch.randint(0, 3, (N * A,), device="cuda", generator=g, dtype=torch.int32)) for _ in range(64)]
        for arm in arms:
            for t in range(args.warmup):
                arm.step(*acts[t % 64], False)
        torch.cuda.synchronize()
        # 1. steps on which no instance reaches the limit: the three arms hold the same games, step for step, so the
        #    per-repeat differences to bare `step` are the cost of the bookkeeping (host: the round trip; device: the launches)
        dev_ms, host_ms = _timed(arms, acts, args.warmup, args.repeats, args.steps)
        for arm in arms:
            d, h = dev_ms[arm.name], host_ms[arm.name]
            diff = [(x - y) * 1e3 for x, y in zip(d, dev_ms["step"])]
            print(json.dumps({"workload": wl, "window": "no_resets", "arm": arm.name, "instances": N, "steps": [args.warmup, quiet_end],
                              "instances_reset": arm.resets if arm.name == "host_composition" else None,
                              "event_ms_per_step": stats(d), "host_ms_per_step": stats(h),
                              "event_us_over_step_same_repeat": stats(diff), **info}), flush=True)
        # 2. a window that contains the step on which every instance reaches number_steps (both resetting arms; bare `step`
        #    would go on with older games from there, so it is left out)
        arms[1].resets = 0
        res = arms[1:]
        for arm in res:
            for t in range(quiet_end, MAX_STEPS - 20):
                arm.step(*acts[t % 64], False)
        dev_ms, host_ms = _timed(res, acts, MAX_STEPS - 20, 2, 40)
        same = bool(torch.equal(res[0].b.obs_tensor(), res[1].b.obs_tensor()) and
                    torch.equal(res[0].b.rewards_tensor(), res[1].b.rewards_tensor()))
        for arm in res:
            print(json.dumps({"workload": wl, "window": "limit_reached", "arm": arm.name, "instances": N,
                              "steps": [MAX_STEPS - 20, MAX_STEPS + 60], "instances_reset": res[0].resets,
                              "event_ms_per_step": stats(dev_ms[arm.name]), "host_ms_per_step": stats(host_ms[arm.name]),
                              "outputs_equal_to_host_composition": same, **info}), flush=True)
        if args.profile:
            from torch.profiler import ProfilerActivity, profile
            os.makedirs(args.profile, exist_ok=True)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for t in range(20):
                    res[1].step(*acts[t % 64], False)
                torch.cuda.synchronize()
            with open(os.path.join(args.profile, f"exp_autoreset_{wl}_kernels.txt"), "w") as f:
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30))
        for arm in arms:
            arm.b.close()


if __name__ == "__main__":
    main()
