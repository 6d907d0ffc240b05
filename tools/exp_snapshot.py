#!/usr/bin/env python
"""What snapshot pools cost on the device: a save of every instance (`k_snapshot` save direction), a restore of every instance
(`k_snapshot` restore direction + the masked `k_obs` behind it), a restore of 5 % of the instances, and, as the baseline, one
`cudaMemcpyAsync` device-to-device (torch's `copy_` of contiguous uint8) of as many bytes as the save writes.

    python tools/exp_snapshot.py [--instances 4096] [--age 2000] [--calls 20] [--repeats 7] [--out FILE]

BASELINE.json configs[1] (arena 1000, 1000 pellets, 25 viruses, 25 bots, tps 4, one 8x128x128 int32 frame), games aged by
`--age` random-walk steps first.  Each repeat times `--calls` back-to-back calls of every arm with device events; the arms
alternate within a repeat and their order rotates between repeats.  A separate torch.profiler pass splits the full restore
into its two kernels.  One JSON line per arm: ms per call (median / min / max over the repeats), bytes read and written per
call (from the slot layout) and the resulting GB/s, plus the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:  # the timing stands without it; say so
        info["power_limit"] = f"unknown ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instances", type=int, default=4096)
    ap.add_argument("--age", type=int, default=2000)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("exp_snapshot.py measures on a GPU; none is visible")
    from agarcl_b200 import make_cfg
    from agarcl_b200.batch import Batch
    N = a.instances
    b = Batch(make_cfg(n_instances=N))
    b.seed(2024)
    b.reset()
    g = torch.Generator(device="cuda").manual_seed(1)
    dxdy = torch.empty((N, 2), device="cuda")
    act = torch.zeros(N, dtype=torch.int32, device="cuda")
    for _ in range(a.age):
        dxdy.uniform_(-1, 1, generator=g)
        act.random_(0, 3, generator=g)
        b.set_actions_device(dxdy.data_ptr(), act.data_ptr())
        b.step()
    torch.cuda.synchronize()
    sb, S = b.slot_bytes, b.layout.stride
    pool = b.snapshot_pool(N)
    every = torch.arange(N, dtype=torch.int32, device="cuda")
    few = torch.full((N,), -1, dtype=torch.int32, device="cuda")
    n_few = max(1, N // 20)
    few[torch.randperm(N, device="cuda", generator=g)[:n_few]] = torch.arange(n_few, dtype=torch.int32, device="cuda")
    dst = torch.empty(N * sb, dtype=torch.uint8, device="cuda")
    src = torch.empty(N * sb, dtype=torch.uint8, device="cuda")
    b.save_states(pool, every)
    torch.cuda.synchronize()
    obs_img = b.obs_shape[1] * b.obs_shape[2] * b.obs_shape[3] * 4 * b.A
    arms = {
        # (call, bytes read, bytes written) per call: a save reads the blobs and writes whole slots; a restore reads the slot
        # headers and blobs and writes the blobs, and its k_obs reads the state and writes one frame per agent
        "save_all": (lambda: b.save_states(pool, every), N * S, N * sb),
        "restore_all": (lambda: b.restore_states(pool, every), N * (64 + S) + N * S, N * S + N * obs_img),
        "restore_5pct": (lambda: b.restore_states(pool, few), n_few * (64 + S) + n_few * S, n_few * S + n_few * obs_img),
        "memcpy_same_bytes": (lambda: dst.copy_(src), N * sb, N * sb),
    }
    for fn, _, _ in arms.values():  # warm-up: every kernel loaded
        fn()
    torch.cuda.synchronize()
    names = list(arms)
    times = {k: [] for k in names}
    for r in range(a.repeats):
        order = names[r % len(names):] + names[:r % len(names)]
        for k in order:
            fn = arms[k][0]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.calls):
                fn()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / a.calls)
    # the two kernels of a full restore, from a profiler pass of their own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.calls):
            b.restore_states(pool, every)
        torch.cuda.synchronize()
    split = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            for k in ("k_snapshot", "k_obs"):
                if k in e.name:
                    split.setdefault(k, []).append(getattr(e, "device_time", None) or e.cuda_time)
    info = gpu_info()
    lines = []
    for k in names:
        t = times[k]
        rd, wr = arms[k][1], arms[k][2]
        med = statistics.median(t)
        lines.append(dict(arm=k, instances=N, age=a.age, slot_bytes=sb, blob_bytes=S, calls=a.calls, repeats=a.repeats,
                          ms_median=round(med, 4), ms_min=round(min(t), 4), ms_max=round(max(t), 4), bytes_read=rd, bytes_written=wr,
                          gb_per_s=round((rd + wr) / med / 1e6, 1), **info))
    lines.append(dict(arm="restore_all_split", instances=N, **{f"{k}_ms_median": round(statistics.median(v) / 1000.0, 4) for k, v in split.items()},
                      **{f"{k}_launches": len(v) for k, v in split.items()}, **info))
    ratio = statistics.median(times["save_all"]) / statistics.median(times["memcpy_same_bytes"])
    lines.append(dict(arm="summary", save_over_memcpy=round(ratio, 3),
                      restore5_over_restore_all=round(statistics.median(times["restore_5pct"]) / statistics.median(times["restore_all"]), 3),
                      **info))
    text = "\n".join(json.dumps(x) for x in lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
    b.close()


if __name__ == "__main__":
    main()
