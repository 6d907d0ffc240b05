#!/usr/bin/env python
"""What the Go-Explore cell archive costs on the device (agarcl_batch_set_archive), on BATCH-sized games.

    python tools/exp_archive.py [--instances 4096] [--age 2000] [--cells 16] [--slots 4096] [--calls 20] [--repeats 7] [--out FILE]

BASELINE.json configs[1] games aged by `--age` random-walk steps, 500-step episodes, device events (exp_common.time_arms: the
arms alternate within a repeat and their order rotates between repeats).

Steps where nothing resets: `step_autoreset` of three identically aged batches, one without an archive, one with an archive
and select = 0, one with select = 1.  The archive adds k_archive_cells, k_archive_commit, the save (k_snapshot, one CTA per
instance, those of the non-winners exit at once) and at the reset k_archive_base, k_archive_select (exits when nothing
resets) and k_start_states.

The step on which all instances reset: every call first restores the same aged games with a step count of 1 under a step limit
of 1 (restore_states), so the step that follows resets every instance.  Arms: no archive (a fresh spawn), an archive with
select = 0 (spawns), and with select = 1 (every instance starts from a drawn entry of a filled archive).

One JSON line per arm: ms per call (median / min / max over the repeats), plus the GPU's name and power limit read in the same
run, and the archive's counters at the end."""
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
    ap.add_argument("--cells", type=int, default=16)
    ap.add_argument("--slots", type=int, default=4096)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("exp_archive.py measures on a GPU; none is visible")
    N = a.instances
    if 1 + a.calls * a.repeats >= 500:
        sys.exit("calls * repeats must stay below the 500-step episode: the quiet steps must not reach the limit")
    plain, sel0, sel1 = (aged_configs1(N, a.age) for _ in range(3))
    for b, _, _ in (plain, sel0, sel1):
        b.set_autoreset(500)
    pools = {}
    for (b, _, _), select in ((sel0, False), (sel1, True)):
        pools[select] = b.snapshot_pool(a.slots)
        b.set_archive(pools[select], a.cells, select=select, seed=1)
    info = gpu_info()
    lines = []

    def autoreset_step(batch):
        b, _, walk = batch

        def f():
            walk.next()
            b.set_actions_device(walk.dxdy.data_ptr(), walk.act.data_ptr())
            b.step_autoreset()
        return f

    quiet = time_arms({"no_archive": autoreset_step(plain), "archive_select0": autoreset_step(sel0),
                       "archive_select1": autoreset_step(sel1)}, a.calls, a.repeats)
    torch.cuda.synchronize()
    counters = {k: sel[0].archive()["counters"].cpu().numpy().tolist() for k, sel in (("select0", sel0), ("select1", sel1))}
    for k, t in quiet.items():
        lines.append(dict(part="quiet_step", arm=k, instances=N, age=a.age, cells=a.cells, slots=a.slots, calls=a.calls,
                          repeats=a.repeats, **stats(t, "ms_"), counters=counters, **info))
    # the step on which every instance resets: the same aged games, restored with step count 1 under a step limit of 1
    every = torch.arange(N, dtype=torch.int32, device="cuda")
    for b, _, _ in (plain, sel0, sel1):
        b.set_autoreset(1)
    plain[0].step_autoreset()
    aged = plain[0].snapshot_pool(N)
    plain[0].save_states(aged, every)
    torch.cuda.synchronize()

    def restored_step(b):
        def f():
            b.restore_states(aged, every)
            b.step_autoreset()
        return f

    full = time_arms({"no_archive": restored_step(plain[0]), "archive_select0": restored_step(sel0[0]),
                      "archive_select1": restored_step(sel1[0])}, a.calls, a.repeats)
    torch.cuda.synchronize()
    assert bool(plain[0].episode()["reset_mask"].all()) and bool((sel1[0].start_result() == 1).all())
    for k, t in full.items():
        lines.append(dict(part="all_reset_step", arm=k, instances=N, age=a.age, cells=a.cells, slots=a.slots, calls=a.calls,
                          repeats=a.repeats, **stats(t, "ms_"), **info))
    write_lines(lines, a.out)
    for b, _, _ in (plain, sel0, sel1):
        b.close()


if __name__ == "__main__":
    main()
