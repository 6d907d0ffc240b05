#!/usr/bin/env python
"""Records a few environments of a BatchedAgarioEnv playing random actions as a video of pictures drawn on the device.

    python tools/record_video.py [--envs 256] [--record 0 1 2 3] [--steps 300] [--size 256] [--view arena|agent] [--out DIR]

Every step draws the chosen environments into slice t of one preallocated device buffer [steps, n, size, size, 3] on the
stream the steps run on, so the loop never waits for the device.  The buffer is copied to the host once at the end and
written per recorded picture as an animated PNG when Pillow imports, else as one .npy array [steps, size, size, 3]."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=256)
    ap.add_argument("--record", type=int, nargs="+", default=[0, 1, 2, 3])
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--view", default="arena", choices=["arena", "agent"])
    ap.add_argument("--num-agents", type=int, default=1)
    ap.add_argument("--fps", type=int, default=15)
    ap.add_argument("--out", default="videos")
    a = ap.parse_args()
    import numpy as np
    import torch
    from agarcl_b200.gym_env import BatchedAgarioEnv
    env = BatchedAgarioEnv(a.envs, num_agents=a.num_agents, num_bots=25, num_viruses=25)
    env.seed(0)
    env.reset()
    ids = torch.tensor(a.record, dtype=torch.int32, device="cuda")
    n = len(a.record) * (a.num_agents if a.view == "agent" else 1)
    video = torch.empty((a.steps, n, a.size, a.size, 3), dtype=torch.uint8, device="cuda")
    NA = a.envs * a.num_agents
    g = torch.Generator(device="cuda").manual_seed(0)
    dxdy = torch.empty((NA, 2), device="cuda")
    act = torch.empty(NA, dtype=torch.int32, device="cuda")
    for t in range(a.steps):
        dxdy.uniform_(-1, 1, generator=g)
        act.random_(0, 3, generator=g)
        env.step(dxdy, act)
        env.render(ids, size=a.size, view=a.view, out=video[t])
    frames = video.cpu().numpy()  # the one wait
    os.makedirs(a.out, exist_ok=True)
    try:
        from PIL import Image
    except ImportError:
        Image = None
    for k in range(n):
        name = os.path.join(a.out, f"{a.view}_{k:03d}")
        if Image is not None:
            imgs = [Image.fromarray(f) for f in frames[:, k]]
            imgs[0].save(name + ".png", save_all=True, append_images=imgs[1:], duration=int(1000 / a.fps), loop=0)
            print(name + ".png")
        else:
            np.save(name + ".npy", frames[:, k])
            print(name + ".npy")
    env.close()


if __name__ == "__main__":
    main()
