"""agarcl_b200 — B200-native batched AgarCL simulator (hot path of machado-research/AgarCL).

Public surface:
  Batch                      owner of a C-ABI batch handle (N lockstep instances on one GPU)
  GridEnvironment            drop-in for agarcl.GridEnvironment (environment/bindings.cpp:99-135), N = 1
  BatchedGridEnvironment     the same interface over N instances, device tensors out
  make_cfg / Cfg / Layout    configuration records of include/agarcl_b200.h
  task_bits                  cfg.task_modes of a list of modes (mixed-task batches: Batch.set_tasks / tasks)
  snapshot_slot_bytes        bytes of one slot of a snapshot pool (Batch.snapshot_pool / save_states / restore_states)
  BOT_HUNGRY .. BOT_AGGRESSIVE_SHY, BOT_TYPES   the built-in bot policies an agent can be driven by (Batch.bot_actions)
"""
from ._abi import Cfg, Layout, StateView, make_cfg, task_bits, OBS_I16, OBS_I32, RNG_MT19937, RNG_PHILOX, RNG_REPLAY  # noqa: F401
from ._abi import BOT_HUNGRY, BOT_HUNGRY_SHY, BOT_AGGRESSIVE, BOT_AGGRESSIVE_SHY, BOT_TYPES  # noqa: F401
from ._lib import snapshot_slot_bytes  # noqa: F401


def __getattr__(name):
    if name == "Batch":
        from .batch import Batch
        return Batch
    if name in ("GridEnvironment", "BatchedGridEnvironment"):
        from . import env
        return getattr(env, name)
    raise AttributeError(name)
