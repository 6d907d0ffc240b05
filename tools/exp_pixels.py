#!/usr/bin/env python
"""What the pixel observation (cfg.pixel_obs, k_draw_views) costs on the device, on BATCH configs[1] games (arena 1000, 1000
pellets, 25 viruses, 25 bots, tps 4, one agent per instance) aged by `--age` random-walk steps:
  views_64, views_128      every agent view (one per instance) at 64 x 64 / 128 x 128 with k_draw_views (agarcl_batch_draw)
  autoreset_pixels128      ms per env-step of step_autoreset with the pixel observation at 128 x 128
  autoreset_grid           ms per env-step of step_autoreset with the grid observation (128 x 128 x 7 int32)
  autoreset_ram_only       ms per env-step of step_autoreset with ram_obs = 2 (no grid frame, no picture)
The three step arms use batches of their own, created, seeded and aged alike, with set_autoreset(500).

    python tools/exp_pixels.py [--instances 4096] [--age 2000] [--calls 20] [--repeats 5] [--out FILE]

Each repeat times `--calls` back-to-back calls of every arm with device events; the arms alternate, their order rotating
between repeats.  One JSON line per arm: ms per call (median / min / max over the repeats), and for the drawing arms the bytes
written and GB/s, with the GPU's name and power limit read in the same run."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from exp_common import RandomWalk, aged_configs1, gpu_info, stats, time_arms, write_lines  # noqa: E402


def aged_autoreset(n, age, **cfg):
    """a configs[1] batch with the extra make_cfg keywords `cfg`, aged like aged_configs1, then stepped by step_autoreset"""
    import torch
    from agarcl_b200 import make_cfg
    from agarcl_b200.batch import Batch
    b = Batch(make_cfg(n_instances=n, **cfg))
    b.seed(2024)
    b.reset()
    b.set_autoreset(500)
    walk = RandomWalk(n)

    def step():
        walk.next()
        b.set_actions_device(walk.dxdy.data_ptr(), walk.act.data_ptr())
        b.step_autoreset()

    for _ in range(age):
        step()
    torch.cuda.synchronize()
    return b, step


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
        sys.exit("exp_pixels.py measures on a GPU; none is visible")
    N = a.instances
    b, _, _ = aged_configs1(N, a.age)
    bufs = {f"views_{S}": torch.empty((N * b.A, S, S, 3), dtype=torch.uint8, device="cuda") for S in (64, 128)}
    arms = {name: (lambda S=buf.shape[1], out=buf: b.draw(None, S, "agent", out=out)) for name, buf in bufs.items()}
    times = time_arms(arms, a.calls, a.repeats)
    b.close()
    steps = {}
    for name, cfg in (("autoreset_pixels128", dict(pixel_obs=128)), ("autoreset_grid", {}), ("autoreset_ram_only", dict(ram_obs=2))):
        steps[name] = aged_autoreset(N, a.age, **cfg)
    times.update(time_arms({k: v[1] for k, v in steps.items()}, a.calls, a.repeats))
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
