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
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from exp_common import aged_configs1, gpu_info, stats, time_arms, write_lines  # noqa: E402


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
    N = a.instances
    b, _, walk = aged_configs1(N, a.age)
    sb, S = b.slot_bytes, b.layout.stride
    pool = b.snapshot_pool(N)
    every = torch.arange(N, dtype=torch.int32, device="cuda")
    few = torch.full((N,), -1, dtype=torch.int32, device="cuda")
    n_few = max(1, N // 20)
    few[torch.randperm(N, device="cuda", generator=walk.g)[:n_few]] = torch.arange(n_few, dtype=torch.int32, device="cuda")
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
    times = time_arms({k: v[0] for k, v in arms.items()}, a.calls, a.repeats)
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
    for k, t in times.items():
        rd, wr = arms[k][1], arms[k][2]
        lines.append(dict(arm=k, instances=N, age=a.age, slot_bytes=sb, blob_bytes=S, calls=a.calls, repeats=a.repeats,
                          **stats(t, "ms_"), bytes_read=rd, bytes_written=wr, gb_per_s=round((rd + wr) / statistics.median(t) / 1e6, 1),
                          **info))
    lines.append(dict(arm="restore_all_split", instances=N, **{f"{k}_ms_median": round(statistics.median(v) / 1000.0, 4) for k, v in split.items()},
                      **{f"{k}_launches": len(v) for k, v in split.items()}, **info))
    ratio = statistics.median(times["save_all"]) / statistics.median(times["memcpy_same_bytes"])
    lines.append(dict(arm="summary", save_over_memcpy=round(ratio, 3),
                      restore5_over_restore_all=round(statistics.median(times["restore_5pct"]) / statistics.median(times["restore_all"]), 3),
                      **info))
    write_lines(lines, a.out)
    b.close()


if __name__ == "__main__":
    main()
