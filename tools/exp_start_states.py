#!/usr/bin/env python
"""What start states cost on the device (agarcl_batch_set_start_states), on BATCH-sized games.

    python tools/exp_start_states.py [--instances 4096] [--age 2000] [--calls 20] [--repeats 7] [--out FILE]

BASELINE.json configs[1] games aged by `--age` random-walk steps, 500-step episodes, device events (exp_common.time_arms: the
arms alternate within a repeat and their order rotates between repeats).

Steps where nothing resets: `step_autoreset` of three identically aged batches, one without a table, one with a table of all -1,
one with a table of slots.  A table adds one mostly-empty launch per step (k_snapshot's start mode, one CTA per instance, none
of which is reset).

The step on which all instances reset: every call first restores the same aged games with a step count of 1 under a step limit
of 1 (restore_states), so the step that follows resets every instance.  Arms: a fresh spawn (no table), start states (a table
of slots), the manual composition it replaces (step_autoreset, then restore_states of the same slots), and the restore plus a
step without any reset, which the other arms' costs are given over (`reset_ms` = arm - that).

One JSON line per arm: ms per call (median / min / max over the repeats), plus the GPU's name and power limit read in the same
run."""
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
        sys.exit("exp_start_states.py measures on a GPU; none is visible")
    N = a.instances
    if 1 + a.calls * a.repeats >= 500:
        sys.exit("calls * repeats must stay below the 500-step episode: the quiet steps must not reach the limit")
    every = torch.arange(N, dtype=torch.int32, device="cuda")
    none = torch.full((N,), -1, dtype=torch.int32, device="cuda")
    plain, minus1, slots = (aged_configs1(N, a.age) for _ in range(3))
    pool = plain[0].snapshot_pool(N)
    plain[0].save_states(pool, every)
    for (b, _, _), table in ((plain, None), (minus1, none), (slots, every)):
        b.set_autoreset(500)
        if table is not None:
            b.set_start_states(pool, table)
    info = gpu_info()
    lines = []

    def autoreset_step(batch):
        b, _, walk = batch

        def f():
            walk.next()
            b.set_actions_device(walk.dxdy.data_ptr(), walk.act.data_ptr())
            b.step_autoreset()
        return f

    quiet = time_arms({"no_table": autoreset_step(plain), "table_all_minus1": autoreset_step(minus1),
                       "table_of_slots": autoreset_step(slots)}, a.calls, a.repeats)
    torch.cuda.synchronize()
    resets = [int(b.episode()["episode_length"].count_nonzero()) for b, _, _ in (plain, minus1, slots)]
    for k, t in quiet.items():
        lines.append(dict(part="quiet_step", arm=k, instances=N, age=a.age, calls=a.calls, repeats=a.repeats, **stats(t, "ms_"),
                          instances_that_ever_reset=resets, **info))
    # the step on which every instance resets: the same aged games, restored with step count 1 under a step limit of 1
    fresh, start = plain[0], slots[0]
    for b in (fresh, start):
        b.set_autoreset(1)
    fresh.step_autoreset()
    aged = fresh.snapshot_pool(N)
    fresh.save_states(aged, every)
    start.set_start_states(aged, every)
    torch.cuda.synchronize()

    def restored_step(b, then_restore=False, autoreset=True):
        def f():
            b.restore_states(aged, every)
            b.step_autoreset() if autoreset else b.step()
            if then_restore:
                b.restore_states(aged, every)
        return f

    full = time_arms({"fresh_spawn": restored_step(fresh), "start_states": restored_step(start),
                      "manual_autoreset_then_restore": restored_step(fresh, then_restore=True),
                      "restore_and_step_without_reset": restored_step(fresh, autoreset=False)}, a.calls, a.repeats)
    torch.cuda.synchronize()
    assert bool((start.start_result() == 1).all()) and bool(fresh.episode()["reset_mask"].all())
    base = statistics.median(full["restore_and_step_without_reset"])
    for k, t in full.items():
        lines.append(dict(part="all_reset_step", arm=k, instances=N, age=a.age, calls=a.calls, repeats=a.repeats, **stats(t, "ms_"),
                          reset_ms=statistics.median(t) - base, **info))
    write_lines(lines, a.out)
    for b, _, _ in (plain, minus1, slots):
        b.close()


if __name__ == "__main__":
    main()
