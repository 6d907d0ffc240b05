"""Host-side mirror of the reference's `agarcl.GridEnvironment` (environment/bindings.cpp:99-135).

`GridEnvironment` keeps the reference's constructor arguments, method names, argument meaning and
error behaviour, and runs on a size-1 batch of the CUDA library; `BatchedGridEnvironment` is the same
interface over N lockstep instances with device tensors out.  Nothing here computes game logic.

Behavioural notes versus the shipped reference (see DESIGN.md, "quirk decisions"):
  * Q11: with `strict_reference=False` (default) the observation is the frame after the last tick of the
    step (what the reference's comments intend); `strict_reference=True` reproduces the shipped
    frame-index arithmetic (all-zero observation for ticks_per_step != num_frames).
  * Q15: `step()` returns rewards in the reference's own order (iteration order of the player map over
    the non-bot players); `BatchedGridEnvironment` returns them indexed by agent.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._abi import OBS_I16, OBS_I32, RNG_MT19937, RNG_PHILOX, make_cfg, task_bits
from .batch import Batch


class _Base:
    def __init__(self, n_instances, num_agents, ticks_per_step, arena_size, pellet_regen, num_pellets, num_viruses,
                 num_bots, reward_type, c_death, mode_number, rng_mode, strict_reference, device, obs_dtype, instance_base=0,
                 ram_obs=False, task_modes=0, pixel_obs=0):
        self._ctor = dict(n_instances=n_instances, num_agents=num_agents, ticks_per_step=ticks_per_step,
                          arena_size=arena_size, pellet_regen=pellet_regen, num_pellets=num_pellets, num_viruses=num_viruses,
                          num_bots=num_bots, reward_type=reward_type, c_death=c_death, mode_number=mode_number,
                          rng_mode=rng_mode, strict_reference=strict_reference, device=device, obs_dtype=obs_dtype,
                          instance_base=instance_base, ram_obs=ram_obs, task_modes=task_modes, pixel_obs=pixel_obs)
        self._obs_cfg = dict(num_frames=1, grid_size=128, observe_cells=True, observe_others=True, observe_viruses=True,
                             observe_pellets=True)
        self._seeds = None
        self._batch = None
        # validate early, like the reference constructor does (Engine::set_mode throws on a bad mode)
        _lib.make_layout(make_cfg(**self._ctor, **self._obs_cfg))

    def _ensure(self):
        if self._batch is None:
            self._batch = Batch(make_cfg(**self._ctor, **self._obs_cfg))
            self._batch.reset()  # the reference constructor ends with reset() (BaseEnvironment.hpp:66), before any seed() can reach it
            if self._seeds is not None:
                self._batch.seed(self._seeds)  # restarts the draw stream: the next reset() is the seed's first episode
        return self._batch

    def configure_observation(self, config):
        """bindings.cpp:104-114 — dict with num_frames, grid_size, observe_cells/others/viruses/pellets"""
        for k in self._obs_cfg:
            if k in config:
                self._obs_cfg[k] = type(self._obs_cfg[k])(config[k])
        if self._batch is not None:
            self._batch.close()
            self._batch = None

    def observation_shape(self):
        L = _lib.make_layout(make_cfg(**self._ctor, **self._obs_cfg))
        return (self._obs_cfg["num_frames"] * L.obs_channels, self._obs_cfg["grid_size"], self._obs_cfg["grid_size"])

    def close(self):
        if self._batch is not None:
            self._batch.close()
            self._batch = None

    _FATAL_FLAGS = 0x020  # AGARCL_FLAG_REPLAY_EXHAUSTED: the recorded draw stream ran out, spawn points are no longer the reference's

    def _check_flags(self, b):
        """the reference's containers grow without bound; this library's are fixed: tell the user instead of diverging silently"""
        f, names = b.flags()
        if f & self._FATAL_FLAGS:
            raise RuntimeError(f"agarcl_b200: simulator state flags {sorted(names)}: the replayed RNG stream is exhausted "
                               "(raise cfg.cap_replay or use rng_mode=RNG_MT19937 / RNG_PHILOX)")
        if f and f != getattr(self, "_flags_warned", 0):
            import warnings
            self._flags_warned = f
            warnings.warn(f"agarcl_b200: simulator state flags {sorted(names)} (a fixed capacity was reached or a libc rand() "
                          "site of the reference was taken; results may differ from the reference from here on)")

    def render(self):
        raise RuntimeError("OpenGL rendering is out of scope of agarcl_b200 (SURVEY.md section 2, rows 11-13)")

    get_frame = render


class GridEnvironment(_Base):
    """Drop-in for agarcl.GridEnvironment(num_agents, ticks_per_step, arena_size, pellet_regen, num_pellets,
    num_viruses, num_bots, reward_type, c_death, mode_number) — bindings.cpp:102."""

    def __init__(self, num_agents, ticks_per_step, arena_size, pellet_regen, num_pellets, num_viruses, num_bots,
                 reward_type=0, c_death=0, mode_number=0, *, rng_mode=RNG_MT19937, strict_reference=False, device=0, pixel_obs=0):
        super().__init__(1, num_agents, ticks_per_step, arena_size, pellet_regen, num_pellets, num_viruses, num_bots,
                         reward_type, c_death, mode_number, rng_mode, strict_reference, device, OBS_I32, pixel_obs=pixel_obs)
        self.num_agents = num_agents
        self._order_agents = None

    def seed(self, s):
        self._seeds = np.array([s], dtype=np.uint64)
        if self._batch is not None:
            self._batch.seed(self._seeds)

    def reset(self):
        self._ensure().reset()
        self._order_agents = None  # (strict_reference: the player-map order changes from episode to episode, quirk Q3)

    def take_actions(self, actions):
        """list of (dx, dy, action) per agent; wrong length raises like EnvironmentException (BaseEnvironment.hpp:142-144)"""
        if len(actions) != self.num_agents:
            raise RuntimeError(f"Number of actions ({len(actions)}) does not match number of agents ({self.num_agents})")
        dxdy = np.array([[a[0], a[1]] for a in actions], dtype=np.float32)
        act = np.array([int(a[2]) for a in actions], dtype=np.int32)
        self._ensure().set_actions(dxdy, act)

    def step(self):
        b = self._ensure()
        rew = np.zeros(self.num_agents, np.float64)
        b.step()
        import torch
        rew = b.rewards_tensor().cpu().numpy()
        self._check_flags(b)
        if self._order_agents is None:
            L = b.layout
            self._order_agents = [p for p in list(L.order)[:L.P] if p < L.A]
        return [float(rew[p]) for p in self._order_agents]  # quirk Q15: player-map order

    def dones(self):
        return [bool(x) for x in self._ensure().dones_tensor().cpu().numpy()]

    def get_state(self):
        """list of int32 arrays (C, G, G), one fresh copy per agent (bindings.cpp:67-91)"""
        obs = self._ensure().obs_tensor().cpu().numpy()
        return [obs[a].copy() for a in range(self.num_agents)]

    def save_env_state(self, path):
        """BaseEnvironment::save_env_state (BaseEnvironment.hpp:213-318; bound at bindings.cpp:135)"""
        self._ensure().save_env_state(0, path)

    def load_env_state(self, path, lossless=False):
        """BaseEnvironment::load_env_state (BaseEnvironment.hpp:320-343; bound for the GoBigger env, bindings.cpp:374)"""
        self._ensure().load_env_state(0, path, lossless)


# ---- plain-data stand-ins for the info structs agarcl binds (environment/bindings.cpp:181-225,
# GoBiggerEnvironment.hpp:30-107); same attribute and method names
class _Location:
    __slots__ = ("x", "y")

    def __init__(self, x, y):
        self.x, self.y = float(x), float(y)


class _Info:
    def __init__(self, dx, dy, radius, score, velocity=(0.0, 0.0)):
        self.position = _Location(dx, dy)
        self.radius = float(radius)
        self.score = int(score)
        self.velocity = (float(velocity[0]), float(velocity[1]))

    def get_position_x(self):
        return self.position.x

    def get_position_y(self):
        return self.position.y


class FoodInfo(_Info):
    pass


class VirusInfo(_Info):
    pass


class SporeInfo(_Info):
    def __init__(self, dx, dy, radius, score, owner):
        super().__init__(dx, dy, radius, score)
        self.owner = int(owner)


class CloneInfo(_Info):
    def __init__(self, dx, dy, radius, score, velocity, direction, owner):
        super().__init__(dx, dy, radius, score, velocity)
        self.direction = float(direction)
        self.owner = int(owner)
        self.teamId = 0


class GlobalState:
    """GoBiggerEnvironment.hpp:30-71"""

    def __init__(self, width, height, frame_limit, last_frame, team_num):
        self._w, self._h, self._limit, self._last, self._teams = width, height, frame_limit, last_frame, team_num

    def update_last_frame_count(self, n):
        self._last = n

    def get_map_width(self):
        return self._w

    def get_map_height(self):
        return self._h

    def get_frame_limit(self):
        return self._limit

    def get_team_num(self):
        return self._teams

    def __str__(self):
        return f"GlobalState(map_width={self._w}, map_height={self._h}, frame_limit={self._limit}, team_num={self._teams})"


class PlayerState:
    """GoBiggerEnvironment.hpp:109-198, filled from one structured-observation record"""

    def __init__(self, player_id, rec=None):
        from ._abi import (RAM_KC, RAM_KP, RAM_KS, RAM_KV, RAM_OFF_CLONE, RAM_OFF_FOOD, RAM_OFF_SPORE, RAM_OFF_VIRUS)
        self._pid = player_id
        self._food, self._virus, self._spore, self._clone = [], [], [], []
        self._score, self._team = 0.0, ""
        if rec is not None and rec[:4].sum() > 0:
            nf, nv, ns, nc = (int(v) for v in rec[:4])
            self._score = float(rec[4])
            f = rec[RAM_OFF_FOOD:RAM_OFF_FOOD + 4 * RAM_KP].reshape(RAM_KP, 4)
            self._food = [FoodInfo(*f[i]) for i in range(min(nf, RAM_KP))]
            v = rec[RAM_OFF_VIRUS:RAM_OFF_VIRUS + 4 * RAM_KV].reshape(RAM_KV, 4)
            self._virus = [VirusInfo(*v[i]) for i in range(min(nv, RAM_KV))]
            sp = rec[RAM_OFF_SPORE:RAM_OFF_SPORE + 4 * RAM_KS].reshape(RAM_KS, 4)
            self._spore = [SporeInfo(*sp[i], owner=player_id) for i in range(min(ns, RAM_KS))]
            c = rec[RAM_OFF_CLONE:RAM_OFF_CLONE + 8 * RAM_KC].reshape(RAM_KC, 8)
            self._clone = [CloneInfo(c[i][0], c[i][1], c[i][2], c[i][3], (c[i][4], c[i][5]), c[i][6], int(c[i][7]))
                           for i in range(min(nc, RAM_KC))]

    def get_player_id(self):
        return self._pid

    def get_food_infos(self):
        return self._food

    def get_virus_infos(self):
        return self._virus

    def get_spore_infos(self):
        return self._spore

    def get_clone_infos(self):
        return self._clone

    def get_team_name(self):
        return self._team

    def get_score(self):
        return self._score

    def canEject(self):
        return True

    def canSplit(self):
        return True


class PlayerStates:
    def __init__(self, states):
        self._states = dict(states)

    def get_all_player_states(self):
        return self._states

    def get_player_state(self, pid):
        return self._states.setdefault(pid, PlayerState(pid))

    def __str__(self):
        return "PlayerStates:\n" + "".join(
            f"  Player {s.get_player_id()}: score={s.get_score()}, food_seen={len(s.get_food_infos())}, "
            f"virus_seen={len(s.get_virus_infos())}, spores_seen={len(s.get_spore_infos())}, "
            f"no_clone={len(s.get_clone_infos())}, team_name=\"{s.get_team_name()}\"\n" for s in self._states.values())


class GoBiggerEnvironment(GridEnvironment):
    """Drop-in for agarcl.GoBiggerEnvironment(map_width, map_height, frame_limit, num_agents, ticks_per_step, arena_size,
    pellet_regen, num_pellets, num_viruses, num_bots, reward_type, c_death=0, mode_number=0, load_env_snapshot=False,
    agent_view=False) — bindings.cpp:323-374.  get_state() returns [{"global_state", "player_states"}] like
    get_state_goBigger (bindings.cpp:28-47), rebuilt from the device's structured-observation records."""

    def __init__(self, map_width, map_height, frame_limit, num_agents, ticks_per_step, arena_size, pellet_regen, num_pellets,
                 num_viruses, num_bots, reward_type, c_death=0, mode_number=0, load_env_snapshot=False, agent_view=False, *,
                 rng_mode=RNG_MT19937, device=0):
        _Base.__init__(self, 1, num_agents, ticks_per_step, arena_size, pellet_regen, num_pellets, num_viruses, num_bots,
                       reward_type, c_death, mode_number, rng_mode, False, device, OBS_I32, ram_obs=True)
        self.num_agents = num_agents
        self._order_agents = None
        self._global = GlobalState(map_width, map_height, frame_limit, 0, num_agents)
        self._frames = 0

    def reset(self):
        super().reset()
        self._frames = 0

    def step(self):
        rew = super().step()
        self._frames += self.num_agents  # one add_frame per agent per step (GoBiggerEnvironment.hpp:515-521)
        return rew

    def observation_shape(self):
        return (self._frames, self._global.get_map_height(), self._global.get_map_width())  # GoBiggerObservation::shape

    def get_state(self):
        ram = self._ensure().ram_tensor()[0].cpu().numpy()
        states = {p: PlayerState(p, ram[p]) for p in range(ram.shape[0]) if ram[p][:4].sum() > 0}
        return [{"global_state": self._global, "player_states": PlayerStates(states)}]

    def ram(self):
        """the raw records [P, RAM_RECORD] float32 (host copy)"""
        return self._ensure().ram_tensor()[0].cpu().numpy()


class BatchedGridEnvironment(_Base):
    """N lockstep GridEnvironments on one GPU.  step() takes arrays/tensors and returns device tensors:
    obs [N*A, C*frames, G, G], rewards f64 [N*A], dones u8 [N*A].  With ram_obs=True the structured
    observation records [N, P, RAM_RECORD] are produced too (ram()).  tasks=(1, 2, ...) makes a mixed-task batch: every
    instance plays its own mode of that set, mode_number first, and changes it at its next reset (set_tasks).  pixel_obs=S: the
    observation is every agent's RGB picture uint8 [N*A, S, S, 3] (Batch.pixels) instead of the grid frame."""

    def __init__(self, n_instances, num_agents=1, ticks_per_step=4, arena_size=1000, pellet_regen=True, num_pellets=1000,
                 num_viruses=25, num_bots=25, reward_type=1, c_death=0, mode_number=0, *, rng_mode=RNG_PHILOX,
                 strict_reference=False, device=0, obs_dtype=OBS_I32, instance_base=0, ram_obs=False, tasks=None, pixel_obs=0):
        super().__init__(n_instances, num_agents, ticks_per_step, arena_size, pellet_regen, num_pellets, num_viruses,
                         num_bots, reward_type, c_death, mode_number, rng_mode, strict_reference, device, obs_dtype,
                         instance_base, ram_obs, task_bits(tasks) if tasks else 0, pixel_obs)
        self.n_instances = n_instances
        self.num_agents = num_agents

    def seed(self, seeds):
        s = np.asarray(seeds, dtype=np.uint64)
        self._seeds = s if s.ndim else (np.arange(self.n_instances, dtype=np.uint64) + s)
        if self._batch is not None:
            self._batch.seed(self._seeds)

    def reset(self, mask=None, stream=0):
        """all instances, or those with mask != 0: a host array (copied to the device) or a CUDA uint8 / bool tensor of
        n_instances entries (read by the device, no host wait)"""
        b = self._ensure()
        if getattr(mask, "is_cuda", False):
            b.reset_device(mask, stream)
        else:
            b.reset(mask, stream)
        return self._obs(b)

    def _obs(self, b):
        return b.pixels() if self._ctor["pixel_obs"] else b.obs_tensor()

    def step(self, dxdy, act, stream=0):
        """dxdy: [N*A, 2] float32, act: [N*A] int32 — numpy (copied) or CUDA torch tensors (zero-copy)"""
        b = self._ensure()
        b.set_actions(dxdy, act, stream)
        b.step(stream)
        return self._obs(b), b.rewards_tensor(), b.dones_tensor()

    def set_autoreset(self, max_steps=0, final_obs=False, reset=True):
        """enables step_autoreset: max_steps > 0 ends an episode after that many steps (0: continuing), final_obs keeps the
        observation a finished episode ended on, reset=False keeps the bookkeeping (done with the step limit, step counters)
        without resetting anything"""
        self._ensure().set_autoreset(max_steps, final_obs, reset)

    def step_autoreset(self, dxdy, act, stream=0):
        """step() followed, on the device, by the episode bookkeeping and the reset of every instance with a done agent;
        returns obs, rewards and the done flags with the step limit folded in (u8 [N*A]); episode() has the rest"""
        b = self._ensure()
        b.set_actions(dxdy, act, stream)
        b.step_autoreset(stream)
        return self._obs(b), b.rewards_tensor(), b.episode()["done"]

    def episode(self):
        return self._ensure().episode()

    def snapshot_pool(self, slots):
        """a zeroed snapshot pool of `slots` slots on the device (Batch.snapshot_pool)"""
        return self._ensure().snapshot_pool(slots)

    def save_states(self, pool, src, slots=None, stream=0):
        """pool slot slots[k] (None: k) <- instance src[k] (Batch.save_states)"""
        self._ensure().save_states(pool, src, slots, stream)

    def restore_states(self, pool, slot_of, stream=0):
        """instance i <- pool slot slot_of[i] where >= 0; returns the result u8 [N] (Batch.restore_states)"""
        return self._ensure().restore_states(pool, slot_of, stream)

    def set_start_states(self, pool, start_slot=None, stream=0):
        """every reset of instance i with start_slot[i] >= 0 begins in pool slot start_slot[i] (Batch.set_start_states); pool
        None: every reset spawns"""
        self._ensure().set_start_states(pool, start_slot, stream)

    def set_archive(self, pool, cells_per_side=None, agent=0, select=True, seed=0):
        """attaches a Go-Explore cell archive whose entries are the slots of `pool` (Batch.set_archive); pool None detaches it"""
        self._ensure().set_archive(pool, cells_per_side, agent, select, seed)

    def archive(self):
        """device views of the archive (Batch.archive)"""
        return self._ensure().archive()

    def set_tasks(self, mode, max_steps=None, stream=0):
        """the task each instance's next reset plays; returns the result u8 [N] (Batch.set_tasks)"""
        return self._ensure().set_tasks(mode, max_steps, stream)

    def tasks(self):
        """device views of the current and pending task of every instance (Batch.tasks)"""
        return self._ensure().tasks()

    def set_task_sizes(self, num_bots=None, num_pellets=None, num_viruses=None, stream=0):
        """the game sizes each instance's next reset plays, at most the constructor's counts; returns the result u8 [N]
        (Batch.set_task_sizes)"""
        return self._ensure().set_task_sizes(num_bots, num_pellets, num_viruses, stream)

    def task_sizes(self):
        """device views of the current and pending game sizes of every instance (Batch.task_sizes)"""
        return self._ensure().task_sizes()

    def bot_actions(self, types, out=None, target=None):
        """(dxdy, act, status) of a built-in bot policy for every agent, on the device (Batch.bot_actions); dxdy and act go
        straight into step()"""
        return self._ensure().bot_actions(types, out, target)

    def ram(self):
        return self._ensure().ram_tensor()

    def flags(self):
        """(OR over all instances, {AGARCL_FLAG name: instances}): a fixed capacity was hit / a non-replayable reference path taken"""
        return self._ensure().flags()

    @property
    def batch(self):
        return self._ensure()
