"""ctypes / numpy mirror of include/agarcl_b200.h (structs, record dtypes, constants).

Nothing here computes: it only describes the C-ABI so Python can talk to
libagarcl_b200.so (product) and, in tests, to oracle/liboracle.so and
oracle/_ref/libagarcl_ref.so (checkers).
"""
import ctypes as C

import numpy as np

MAX_CELLS = 32
VET_CAP = 16
MAX_PLAYERS = 64

FLAG_NAMES = {
    0x001: "FOOD_OVERFLOW", 0x002: "VIRUS_OVERFLOW", 0x004: "CELL_OVERFLOW", 0x008: "VET_OVERFLOW",
    0x010: "EATER_OVERFLOW", 0x020: "REPLAY_EXHAUSTED", 0x040: "PCD_TIE", 0x080: "RAND_SITE",
    0x100: "MASS_LUT", 0x200: "REMOVE_OVERFLOW",
}

RNG_PHILOX, RNG_REPLAY, RNG_MT19937 = 0, 1, 2
# structured ("ram") observation record, include/agarcl_b200.h
RAM_HDR, RAM_KP, RAM_KV, RAM_KS, RAM_KC = 8, 192, 16, 32, 32
RAM_OFF_FOOD = RAM_HDR
RAM_OFF_VIRUS = RAM_OFF_FOOD + 4 * RAM_KP
RAM_OFF_SPORE = RAM_OFF_VIRUS + 4 * RAM_KV
RAM_OFF_CLONE = RAM_OFF_SPORE + 4 * RAM_KS
RAM_RECORD = RAM_OFF_CLONE + 8 * RAM_KC
OBS_I32, OBS_I16 = 0, 1
DRAW_VIEWS = {"arena": 0, "agent": 1}  # AGARCL_DRAW_ARENA, AGARCL_DRAW_AGENT
# built-in bot policies (agarcl_batch_bot_actions): AGARCL_BOT_* bot types and per-agent results
BOT_HUNGRY, BOT_HUNGRY_SHY, BOT_AGGRESSIVE, BOT_AGGRESSIVE_SHY = 0, 1, 2, 3
BOT_TYPES = {"hungry": BOT_HUNGRY, "hungry_shy": BOT_HUNGRY_SHY, "aggressive": BOT_AGGRESSIVE, "aggressive_shy": BOT_AGGRESSIVE_SHY}
BOT_SKIPPED, BOT_DECIDED, BOT_NO_PELLET, BOT_DEAD, BOT_BAD_TYPE = 0, 1, 2, 3, 4


class Cfg(C.Structure):
    """struct agarcl_cfg"""
    _fields_ = [(n, C.c_int32) for n in (
        "n_instances",
        "num_agents", "ticks_per_step", "arena_size", "pellet_regen", "num_pellets", "num_viruses", "num_bots",
        "reward_type", "c_death", "mode_number",
        "num_frames", "grid_size", "observe_cells", "observe_others", "observe_viruses", "observe_pellets",
        "obs_dtype", "strict_reference", "rng_mode",
        "cap_viruses", "cap_foods", "cap_replay", "device", "instance_base", "ram_obs", "task_modes", "pixel_obs")]


class Layout(C.Structure):
    """struct agarcl_layout"""
    _fields_ = [(n, C.c_int32) for n in ("P", "A", "cap_cells", "cap_pellets", "cap_viruses", "cap_foods", "cap_replay")] + \
               [(n, C.c_uint32) for n in ("off_hdr", "off_players", "off_cells", "off_viruses", "off_foods", "off_pellets", "stride")] + \
               [(n, C.c_int32) for n in ("mass_decay", "squared_pellets", "regen", "agent_mass", "obs_channels")] + \
               [("order", C.c_int32 * MAX_PLAYERS), ("bot_type", C.c_int32 * MAX_PLAYERS)]


class ArchiveCfg(C.Structure):
    """struct agarcl_archive_cfg"""
    _fields_ = [(n, C.c_int32) for n in ("cells_per_side", "agent", "select", "pad")] + [("seed", C.c_uint64)]


class Archive(C.Structure):
    """struct agarcl_archive"""
    _fields_ = [(n, C.c_void_p) for n in ("cell_of", "base_score", "base_length", "key_entry", "visits", "entry_key", "entry_score",
                                          "entry_length", "entry_chosen", "counters")] + [("keys", C.c_int64), ("entries", C.c_int64)]


CELL_DT = np.dtype([("x", "<f4"), ("y", "<f4"), ("vx", "<f4"), ("vy", "<f4"), ("svx", "<f4"), ("svy", "<f4"),
                    ("mass", "<u4"), ("id", "<u4"), ("recomb_tick", "<u4"), ("pad", "<u4", (3,))])
VIRUS_DT = np.dtype([("x", "<f4"), ("y", "<f4"), ("mass", "<u4"), ("hits", "<i4"), ("vx", "<f4"), ("vy", "<f4"),
                     ("pad", "<u4", (2,))])
FOOD_DT = np.dtype([("x", "<f4"), ("y", "<f4"), ("vx", "<f4"), ("vy", "<f4")])
PELLET_DT = np.dtype([("x", "<f4"), ("y", "<f4")])
PLAYER_DT = np.dtype([("n_cells", "<i4"), ("target_x", "<f4"), ("target_y", "<f4"), ("action", "<i4"),
                      ("split_cd", "<i4"), ("feed_cd", "<i4"), ("anti_team_decay", "<f4"),
                      ("elapsed_ticks", "<i4"), ("last_decay_tick", "<i4"), ("bot_type", "<i4"),
                      ("min_mass_cell", "<u4"), ("food_eaten", "<i4"), ("highest_mass", "<u4"),
                      ("cells_eaten", "<i4"), ("viruses_eaten", "<i4"), ("vet_count", "<i4"),
                      ("vet_ticks", "<i4", (VET_CAP,))])
HDR_DT = np.dtype([("tick", "<u4"), ("next_cell_id", "<u4"), ("n_pellets", "<i4"), ("n_viruses", "<i4"),
                   ("n_foods", "<i4"), ("rng_cursor", "<u4"), ("flags", "<u4"), ("seed_lo", "<u4"),
                   ("seed_hi", "<u4"), ("done_sticky", "<u4"), ("respawned_lo", "<u4"), ("respawned_hi", "<u4"),
                   ("pad", "<u4", (4,))])

assert CELL_DT.itemsize == 48 and VIRUS_DT.itemsize == 32 and FOOD_DT.itemsize == 16
assert PELLET_DT.itemsize == 8 and PLAYER_DT.itemsize == 128 and HDR_DT.itemsize == 64


def make_cfg(n_instances=1, num_agents=1, ticks_per_step=4, arena_size=1000, pellet_regen=True,
             num_pellets=1000, num_viruses=25, num_bots=25, reward_type=1, c_death=0, mode_number=0,
             num_frames=1, grid_size=128, observe_cells=True, observe_others=True, observe_viruses=True,
             observe_pellets=True, obs_dtype=OBS_I32, strict_reference=False, rng_mode=RNG_PHILOX,
             cap_viruses=0, cap_foods=0, cap_replay=0, device=0, instance_base=0, ram_obs=False, task_modes=0, pixel_obs=0):
    """task_modes: 0, or the bit mask of the modes a mixed-task batch may run (include/agarcl_b200.h); task_bits() makes one
    from a list of modes.  pixel_obs: 0, or the size S of the pixel observation (one RGB picture [S, S, 3] per agent after every
    step and reset instead of the grid frame)"""
    c = Cfg()
    for k, v in list(locals().items()):
        if k in ("c",):
            continue
        setattr(c, k, int(v))
    return c


def task_bits(modes):
    """bit mask (cfg.task_modes) of an iterable of mode numbers"""
    bits = 0
    for m in modes:
        m = int(m)
        if not 0 <= m <= 10:
            raise ValueError(f"mode {m} is outside 0..10")
        bits |= 1 << m
    return bits


class StateView:
    """Named numpy views over one instance blob (uint8 array of layout.stride bytes)."""

    def __init__(self, layout, blob=None):
        self.layout = layout
        self.blob = np.zeros(layout.stride, dtype=np.uint8) if blob is None else blob
        assert self.blob.dtype == np.uint8 and self.blob.size == layout.stride
        L, b = layout, self.blob
        self.hdr = b[L.off_hdr:L.off_hdr + 64].view(HDR_DT)[0]
        self.players = b[L.off_players:L.off_players + 128 * L.P].view(PLAYER_DT)
        self.cells = b[L.off_cells:L.off_cells + 48 * L.P * L.cap_cells].view(CELL_DT).reshape(L.P, L.cap_cells)
        self.viruses = b[L.off_viruses:L.off_viruses + 32 * L.cap_viruses].view(VIRUS_DT)
        self.foods = b[L.off_foods:L.off_foods + 16 * L.cap_foods].view(FOOD_DT)
        self.pellets = b[L.off_pellets:L.off_pellets + 8 * L.cap_pellets].view(PELLET_DT)

    def copy(self):
        return StateView(self.layout, self.blob.copy())

    @property
    def ptr(self):
        return self.blob.ctypes.data_as(C.c_void_p)

    def flag_names(self):
        f = int(self.hdr["flags"])
        return [n for bit, n in FLAG_NAMES.items() if f & bit]


def compare_states(a, b, pos_tol=0.0, check_ids=True):
    """Field-by-field comparison of two StateViews. Returns a list of human-readable differences.

    Discrete fields (counts, masses, timers, cooldowns, stats) must be identical; float fields must
    agree bit-for-bit when pos_tol == 0, else within pos_tol absolute.  Cell ids are compared by
    their order inside each player (only relative order is ever used, Engine.hpp:157,176-187).
    NaN == NaN counts as equal.
    """
    diffs = []
    L = a.layout

    def feq(x, y, what):
        x = np.asarray(x, dtype=np.float32)
        y = np.asarray(y, dtype=np.float32)
        if pos_tol == 0.0:
            same = (x.view(np.uint32) == y.view(np.uint32)) | (np.isnan(x) & np.isnan(y)) | ((x == 0) & (y == 0))
        else:
            same = (np.abs(x - y) <= pos_tol) | (np.isnan(x) & np.isnan(y))
        if not np.all(same):
            idx = np.argwhere(~same)[:4].tolist()
            diffs.append(f"{what}: {int((~same).sum())} float mismatches, first at {idx}: "
                         f"{x[~same][:4].tolist()} vs {y[~same][:4].tolist()}")

    def ieq(x, y, what):
        if not np.array_equal(x, y):
            diffs.append(f"{what}: {np.asarray(x).tolist() if np.size(x) < 40 else '...'} vs "
                         f"{np.asarray(y).tolist() if np.size(y) < 40 else '...'}")

    for f in ("tick", "n_pellets", "n_viruses", "n_foods", "done_sticky"):
        ieq(a.hdr[f], b.hdr[f], f"hdr.{f}")
    n = int(min(a.hdr["n_pellets"], b.hdr["n_pellets"]))
    for f in ("x", "y"):
        feq(a.pellets[f][:n], b.pellets[f][:n], f"pellets.{f}")
    n = int(min(a.hdr["n_viruses"], b.hdr["n_viruses"]))
    for f in ("x", "y", "vx", "vy"):
        feq(a.viruses[f][:n], b.viruses[f][:n], f"viruses.{f}")
    for f in ("mass", "hits"):
        ieq(a.viruses[f][:n], b.viruses[f][:n], f"viruses.{f}")
    n = int(min(a.hdr["n_foods"], b.hdr["n_foods"]))
    for f in ("x", "y", "vx", "vy"):
        feq(a.foods[f][:n], b.foods[f][:n], f"foods.{f}")
    for f in ("n_cells", "action", "split_cd", "feed_cd", "elapsed_ticks", "last_decay_tick", "bot_type",
              "min_mass_cell", "food_eaten", "highest_mass", "cells_eaten", "viruses_eaten", "vet_count"):
        ieq(a.players[f], b.players[f], f"players.{f}")
    for f in ("target_x", "target_y", "anti_team_decay"):
        feq(a.players[f], b.players[f], f"players.{f}")
    for p in range(L.P):
        k = int(min(a.players["vet_count"][p], b.players["vet_count"][p], VET_CAP))
        ieq(a.players["vet_ticks"][p][:k], b.players["vet_ticks"][p][:k], f"players[{p}].vet_ticks")
        n = int(min(a.players["n_cells"][p], b.players["n_cells"][p], L.cap_cells))
        ca, cb = a.cells[p][:n], b.cells[p][:n]
        for f in ("x", "y", "vx", "vy", "svx", "svy"):
            feq(ca[f], cb[f], f"cells[{p}].{f}")
        ieq(ca["mass"], cb["mass"], f"cells[{p}].mass")
        # recombine eligibility at the current tick is what is observable
        t = int(a.hdr["tick"])
        ieq(np.maximum(ca["recomb_tick"].astype(np.int64), t), np.maximum(cb["recomb_tick"].astype(np.int64), t),
            f"cells[{p}].recomb_tick")
        if check_ids and n > 1:
            ieq(np.argsort(ca["id"], kind="stable"), np.argsort(cb["id"], kind="stable"), f"cells[{p}].id-order")
    return diffs
