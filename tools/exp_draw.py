#!/usr/bin/env python
"""What pictures of game states cost on the device (agarcl_batch_draw, k_draw), on BATCH configs[1] games (arena 1000, 1000
pellets, 25 viruses, 25 bots, tps 4) aged by `--age` random-walk steps:
  arena16_512   16 arena pictures at 512 x 512
  arena16_1024  16 arena pictures at 1024 x 1024
  agents_128    every agent view (one per instance) at 128 x 128, with the bytes written per second against HBM bandwidth
  step          one Batch.step of the same batch, for scale

    python tools/exp_draw.py [--instances 4096] [--age 2000] [--calls 20] [--repeats 5] [--out FILE]

Each repeat times `--calls` back-to-back calls of every arm with device events; the arms alternate within a repeat.  One JSON
line per arm: ms per call (median / min / max over the repeats), bytes written and GB/s, with the GPU's name and power limit
read in the same run."""
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
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("exp_draw.py measures on a GPU; none is visible")
    N = a.instances
    b, step, _ = aged_configs1(N, a.age)
    src16 = torch.arange(0, N, max(1, N // 16), dtype=torch.int32, device="cuda")[:16].contiguous()
    bufs = {"arena16_512": torch.empty((src16.numel(), 512, 512, 3), dtype=torch.uint8, device="cuda"),
            "arena16_1024": torch.empty((src16.numel(), 1024, 1024, 3), dtype=torch.uint8, device="cuda"),
            "agents_128": torch.empty((N * b.A, 128, 128, 3), dtype=torch.uint8, device="cuda")}
    arms = {"arena16_512": lambda: b.draw(src16, 512, "arena", out=bufs["arena16_512"]),
            "arena16_1024": lambda: b.draw(src16, 1024, "arena", out=bufs["arena16_1024"]),
            "agents_128": lambda: b.draw(None, 128, "agent", out=bufs["agents_128"])}
    # (stepping changes the games pictured: the step is timed after the drawing arms)
    times = time_arms(arms, a.calls, a.repeats)
    times.update(time_arms({"step": step}, a.calls, a.repeats))
    info = gpu_info()
    lines = []
    for name, ts in times.items():
        rec = {"arm": name, "instances": N, "age": a.age, **stats(ts, "ms_")}
        if name in bufs:
            nbytes = bufs[name].numel()
            rec.update(pictures=int(bufs[name].shape[0]), size=int(bufs[name].shape[1]), bytes_written=nbytes,
                       write_GBps=nbytes / (rec["ms_median"] * 1e-3) / 1e9)
        rec.update(info)
        lines.append(rec)
    write_lines(lines, a.out)


if __name__ == "__main__":
    main()
