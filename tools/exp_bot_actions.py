#!/usr/bin/env python
"""What the built-in bot policies for agents cost on the device (agarcl_batch_bot_actions, k_bot_actions), for every agent of
BATCH configs[1] games (arena 1000, 1000 pellets, 25 viruses, 25 bots, tps 4) aged by `--age` random-walk steps, against one
step of the same batch:
  <type>        Batch.bot_actions(type) for every agent, called from Python (what a training loop pays, host overhead included)
  <type>_graph  the same calls replayed from a CUDA graph: the device time of the kernel
  step          one Batch.step, for scale

    python tools/exp_bot_actions.py [--instances 4096] [--age 2000] [--calls 50] [--repeats 5] [--out FILE]

Each repeat times `--calls` back-to-back calls of every arm with device events, after a warm-up; the arms alternate within a
repeat.  One JSON line per arm: ms per call (median / min / max over the repeats), with the GPU's name and power limit read in
the same run."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from exp_common import aged_configs1, gpu_info, stats, time_arms, write_lines  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instances", type=int, default=4096)
    ap.add_argument("--age", type=int, default=2000)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("exp_bot_actions.py measures on a GPU; none is visible")
    from agarcl_b200 import BOT_TYPES
    N = a.instances
    b, step, _ = aged_configs1(N, a.age)
    NA = N * b.A
    out = (torch.empty((NA, 2), device="cuda"), torch.empty(NA, dtype=torch.int32, device="cuda"),
           torch.empty(NA, dtype=torch.uint8, device="cuda"))
    arms = {}
    s = torch.cuda.Stream()
    for name, t in BOT_TYPES.items():
        arms[name] = (lambda t=t: b.bot_actions(t, out=out))
        arms[name]()  # warm-up (and the broadcast type tensor, made once)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            for _ in range(a.calls):
                b.bot_actions(t, out=out)
        arms[name + "_graph"] = graph.replay
    arms["step"] = step
    times = time_arms(arms, a.calls, a.repeats, graphs=[k for k in arms if k.endswith("_graph")])
    status = torch.bincount(out[2].long(), minlength=5).tolist()  # (of the type called last)
    info = gpu_info()
    lines = []
    for name, ts in times.items():
        rec = {"arm": name, "instances": N, "agents": NA, "age": a.age, **stats(ts, "ms_")}
        if name != "step":
            rec["players_per_instance"] = b.layout.P
        rec.update(info)
        lines.append(rec)
    lines.append({"last_status_counts": status})
    write_lines(lines, a.out)


if __name__ == "__main__":
    main()
