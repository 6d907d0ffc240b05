"""What the device measurements of tools/exp_*.py share: the GPU's name and power limit, random-walk actions and the aged
BASELINE.json configs[1] batch they age, the device-event timer that runs the arms alternately, and the JSON-line writer."""
import json
import statistics
import subprocess


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:  # the timing stands without it; say so
        info["power_limit"] = f"not read: {e}"
    return info


class RandomWalk:
    """device actions of n agents, redrawn by next(): dxdy uniform in [-1, 1), act in 0..2, from a generator seeded with 1"""

    def __init__(self, n):
        import torch
        self.g = torch.Generator(device="cuda").manual_seed(1)
        self.dxdy = torch.empty((n, 2), device="cuda")
        self.act = torch.zeros(n, dtype=torch.int32, device="cuda")

    def next(self):
        self.dxdy.uniform_(-1, 1, generator=self.g)
        self.act.random_(0, 3, generator=self.g)


def aged_configs1(n, age):
    """a batch of n BASELINE.json configs[1] instances (seed 2024) aged by `age` random-walk steps; returns the batch, a
    function that takes one more such step, and the walk"""
    import torch
    from agarcl_b200 import make_cfg
    from agarcl_b200.batch import Batch
    b = Batch(make_cfg(n_instances=n))
    b.seed(2024)
    b.reset()
    walk = RandomWalk(n)

    def step():
        walk.next()
        b.set_actions_device(walk.dxdy.data_ptr(), walk.act.data_ptr())
        b.step()

    for _ in range(age):
        step()
    torch.cuda.synchronize()
    return b, step, walk


def time_arms(arms, calls, repeats, graphs=()):
    """ms per call of every arm of {name: fn}, one value per repeat: after one warm-up call of every arm, each repeat records
    `calls` back-to-back calls of every arm between two device events (one call of an arm named in `graphs`: the replay of a
    CUDA graph that holds `calls` of them); the arms run one after the other, their order rotating by one between repeats"""
    import torch
    names = list(arms)
    for f in arms.values():
        f()
    torch.cuda.synchronize()
    ms = {k: [] for k in names}
    for r in range(repeats):
        for k in names[r % len(names):] + names[:r % len(names)]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(1 if k in graphs else calls):
                arms[k]()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1) / calls)
    return ms


def stats(xs, prefix=""):
    """median / min / max of xs, under keys prefixed with `prefix`"""
    return {prefix + "median": statistics.median(xs), prefix + "min": min(xs), prefix + "max": max(xs)}


def write_lines(records, out=None):
    """one JSON line per record on stdout and, with `out`, in that file"""
    text = "\n".join(json.dumps(r) for r in records)
    print(text, flush=True)
    if out:
        with open(out, "w") as f:
            f.write(text + "\n")
