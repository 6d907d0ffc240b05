"""Host-side mirror of the reference's gym wrapper (gym_agario/AgarioEnv.py, gym_agario/__init__.py).

`AgarioEnv` keeps the reference's constructor keywords, action format, return tuples and ids
(`agario-grid-v0`, `agario-gobigger-v0`; `agario-ram-v0` is the flat structured observation the reference's
disabled ram test expects, tests/ram_env_test.py:11,67-92) over a size-1 batch; `BatchedAgarioEnv` is the
vector form over N lockstep instances with device tensors and auto-reset.  gymnasium is used when it is
installed and replaced by minimal stand-ins when it is not (it is absent from the build image).

Deliberate differences from the shipped wrapper, which cannot run as written (SURVEY quirks Q12/Q13/Q17):
  * `_make_environment` references an undefined `args` and passes 11 positional arguments to a 10-argument
    binding (AgarioEnv.py:213-227): here the 10 documented arguments are passed;
  * `kwargs | grid_defaults` lets the defaults override the caller (AgarioEnv.py:226): here the caller wins;
  * the action noise is computed and then discarded (AgarioEnv.py:282-296): no noise is applied here either.
"""
import numpy as np

from .env import BatchedGridEnvironment, GoBiggerEnvironment, GridEnvironment

try:  # pragma: no cover - gymnasium is optional
    import gymnasium as gym
    from gymnasium import spaces
    _EnvBase = gym.Env
except Exception:  # minimal stand-ins with the attributes the wrapper and its users touch
    gym = None

    class _Box:
        def __init__(self, low, high, shape=None, dtype=np.float32):
            self.low, self.high, self.shape, self.dtype = low, high, tuple(shape) if shape is not None else (), np.dtype(dtype)

        def contains(self, x):
            x = np.asarray(x)
            return x.shape == self.shape and bool(np.all(x >= self.low)) and bool(np.all(x <= self.high))

        def sample(self):
            return np.random.uniform(self.low, self.high, size=self.shape).astype(self.dtype)

    class _Discrete:
        def __init__(self, n):
            self.n = n

        def contains(self, x):
            return int(x) == x and 0 <= int(x) < self.n

        def sample(self):
            return int(np.random.randint(self.n))

    class _Tuple(tuple):
        def __new__(cls, items):
            return super().__new__(cls, items)

        def sample(self):
            return tuple(s.sample() for s in self)

    class spaces:  # noqa: N801
        Box, Discrete, Tuple = _Box, _Discrete, _Tuple

    class _EnvBase:
        pass


def _env_args(kwargs):
    """AgarioEnv._get_env_args (AgarioEnv.py:298-363): difficulty presets, overridable one by one"""
    difficulty = kwargs.get("difficulty", "normal").lower()
    if difficulty not in ("normal", "empty", "trivial"):
        raise ValueError(f"Unrecognized difficulty: {difficulty}")
    d = dict(num_agents=1, ticks_per_step=4, arena_size=1000, pellet_regen=True, num_pellets=1000, num_viruses=0, num_bots=0,
             reward_type=1, c_death=0, mode=0)
    if difficulty == "trivial":
        d.update(arena_size=50, num_pellets=200)
    for k in d:
        if k in kwargs:
            d[k] = kwargs[k]
    if type(d["ticks_per_step"]) is not int or d["ticks_per_step"] <= 0:
        raise ValueError("ticks_per_step must be a positive integer")
    return d


_OBS_KEYS = ("num_frames", "grid_size", "observe_cells", "observe_others", "observe_viruses", "observe_pellets")


class AgarioEnv(_EnvBase):
    metadata = {"render_modes": ["human", "rgb_array"], "render_fps": 60}

    def __init__(self, obs_type="grid", render_mode=None, render_size=512, render_view="arena", pixel_size=128, **kwargs):
        if obs_type not in ("ram", "screen", "grid", "gobigger", "pixels"):
            raise ValueError(obs_type)
        if render_view not in ("arena", "agent"):
            raise ValueError(f"render_view must be 'arena' or 'agent', got {render_view!r}")
        if obs_type == "screen":
            raise ValueError("agarcl_b200 does not include ScreenEnvironment (OpenGL, out of scope)")
        a = _env_args(kwargs)
        self.num_agents = a["num_agents"]
        self.multi_agent = bool(kwargs.get("multi_agent", False)) or self.num_agents > 1
        self.obs_type = obs_type
        self.render_mode = render_mode
        self.render_size, self.render_view = int(render_size), render_view
        self.number_of_steps = kwargs.get("number_steps", 500)
        self.mode = a["mode"]
        self.env_type = kwargs.get("env_type", 0)  # 0 episodic, 1 continuing
        self.add_noise = kwargs.get("add_noise", True)
        self.steps = None
        self._seed = None
        pos = (a["num_agents"], a["ticks_per_step"], a["arena_size"], a["pellet_regen"], a["num_pellets"], a["num_viruses"],
               a["num_bots"], a["reward_type"], a["c_death"], a["mode"])
        extra = {k: kwargs[k] for k in ("device", "rng_mode") if k in kwargs}
        if obs_type == "grid":
            self._env = GridEnvironment(*pos, **extra)
            self._env.configure_observation({k: kwargs[k] for k in _OBS_KEYS if k in kwargs})
            c, w, h = self._env.observation_shape()
            self.observation_space = spaces.Box(-1, np.iinfo(np.int32).max, (w, h, c), dtype=np.int32)
        elif obs_type == "pixels":  # every agent's RGB picture, drawn on the device (include/agarcl_b200.h, cfg.pixel_obs)
            S = int(pixel_size)
            self._env = GridEnvironment(*pos, pixel_obs=S, **extra)
            self.observation_space = spaces.Box(0, 255, (S, S, 3), dtype=np.uint8)
        else:
            self._env = GoBiggerEnvironment(kwargs.get("map_width", 512), kwargs.get("map_height", 512),
                                            kwargs.get("frame_limit", 1000), *pos, **extra)
            self._env.configure_observation({k: kwargs[k] for k in _OBS_KEYS if k in kwargs})
            from ._abi import RAM_RECORD
            shape = (RAM_RECORD,) if obs_type == "ram" else self._env.observation_shape()
            self.observation_space = spaces.Box(-1e4 if obs_type == "ram" else 0, 1e6 if obs_type == "ram" else 255, shape,
                                                dtype=np.float32)
        self.action_space = spaces.Tuple((spaces.Box(low=-1, high=1, shape=(2,)), spaces.Discrete(3)))

    # ---- gym API (AgarioEnv.py:77-132)
    def step(self, actions):
        assert self.steps is not None, "Cannot call step() before calling reset()"
        actions = self._sanitize_actions(actions)
        self._env.take_actions(actions)
        rewards = self._env.step()
        assert len(rewards) == self.num_agents
        self.observations = self._make_observations()
        dones = self._env.dones()
        truncations = [False] * len(dones)
        if self.steps >= self.number_of_steps and self.env_type == 0:
            dones = [True] * len(dones)
        if not self.multi_agent:
            self.observations, rewards, dones, truncations = self.observations[0], rewards[0], dones[0], truncations[0]
        self.steps += 1
        return self.observations, rewards, dones, truncations, {"steps": self.steps, "untransformed_rewards": rewards}

    def reset(self, **kwargs):
        self.steps = 0
        self._env.reset()
        obs = self._make_observations()
        return (obs if self.multi_agent else obs[0]), {}

    def seed(self, seed=None):
        if seed is not None:
            self._seed = seed
            self._env.seed(seed)
            return [self._seed]

    def render(self):
        """render_mode "rgb_array": an RGB picture uint8 [render_size, render_size, 3] of the game drawn on the device
        (include/agarcl_b200.h, agarcl_batch_draw) -- the whole arena, or with render_view "agent" the agent's observation
        window ([num_agents, S, S, 3] for a multi-agent environment).  Other render modes need OpenGL, which is out of scope."""
        if self.render_mode != "rgb_array":
            raise RuntimeError("OpenGL rendering is out of scope of agarcl_b200 (render_mode='rgb_array' draws pictures)")
        pics = self._env._ensure().draw(None, self.render_size, self.render_view).cpu().numpy()
        return pics if self.render_view == "agent" and self.multi_agent else pics[0]

    def close(self):
        self._env.close()

    def save_env_state(self, filename):
        self._env.save_env_state(filename)

    def load_env_state(self, filename):
        self._env.load_env_state(filename)

    # ---- helpers
    def _make_observations(self):
        if self.obs_type == "pixels":
            pics = self._env._ensure().pixels().cpu().numpy()
            return [pics[a] for a in range(self.num_agents)]
        if self.obs_type == "grid":
            return [np.transpose(s, [1, 2, 0]) for s in self._env.get_state()]  # NCHW -> HWC view (AgarioEnv.py:192-194)
        if self.obs_type == "ram":
            ram = self._env.ram()
            return [ram[a].copy() for a in range(self.num_agents)]
        states = self._env.get_state()
        return states * self.num_agents if len(states) == 1 and self.num_agents > 1 else states

    def _sanitize_actions(self, actions):
        if not self.multi_agent and type(actions) is not list:
            actions = [actions]
        if type(actions) is not list:
            raise ValueError("Action list must be a list of two-element tuples")
        if len(actions) != self.num_agents:
            raise ValueError(f"Number of actions {len(actions)} does not match number of agents {self.num_agents}")
        out = []
        for tgt, a in actions:
            tgt = np.asarray(tgt, dtype=np.float32)
            if not (self.action_space[0].contains(tgt) and self.action_space[1].contains(a)):
                raise ValueError(f"action {(tgt, a)} not in action space")
            out.append((float(tgt[0]), float(tgt[1]), int(a)))
        return out


class BatchedAgarioEnv:
    """Vector environment: N lockstep instances on one GPU, device tensors in and out, auto-reset on the device.

    step(dxdy [N*A, 2] float32, act [N*A] int32) -> obs, rewards (float32), dones, truncations (bool tensors), info.
    An instance with a done agent, or that reached `number_steps` (episodic, env_type 0), is reset within the same step: its
    observation is the first of the new episode, while the rewards and dones returned are those of the finished step.  The
    host never waits for the device, so step t+1 can be queued while step t runs.  info (device tensors):
      steps           i64 [N]    steps since the instance's last reset
      reset_mask      bool [N]   instances reset by this step
      episode_return  f64 [N*A]  return of the episode an instance just finished (read where reset_mask is set)
      episode_length  i64 [N]    its length in steps (likewise)
      final_obs       the observation that episode ended on (grid: [N*A, C*frames, G, G]; ram: [N, A, RAM_RECORD]; pixels: [N*A,
                      S, S, 3]); only with final_obs=True, which allocates as much device memory again as the observation
    obs, dones and every info tensor are views of library-owned buffers that the next step() overwrites: copy what must
    outlive it.  With auto_reset=False nothing is reset: the step limit is folded into dones, steps keeps counting, and
    info has "steps" only.

    tasks=[1, 2, ...]: a mixed-task batch, every environment plays its own mini-game (mode) of that set -- `mode` (default:
    the first of the list) to begin with -- and set_tasks() chooses what each one plays from its next reset on, with its own
    step limit.  info["task"] (i32 [N]) is then every environment's current mode: after an auto-reset, the new episode's.

    obs_type="pixels": the observation is every agent's RGB picture uint8 [N*A, pixel_size, pixel_size, 3] (HWC), drawn on the
    device after every step from the same moment as the grid observation (include/agarcl_b200.h, cfg.pixel_obs); no grid frame
    is rendered.  Frame stacking is the caller's: info["reset_mask"] says which stacks to clear."""

    def __init__(self, n_envs, obs_type="grid", auto_reset=True, final_obs=False, tasks=None, pixel_size=128, **kwargs):
        if obs_type not in ("grid", "ram", "pixels"):
            raise ValueError(obs_type)
        if tasks and "mode" not in kwargs:
            kwargs = dict(kwargs, mode=int(list(tasks)[0]))
        a = _env_args(kwargs)
        self.n_envs, self.num_agents, self.obs_type, self.auto_reset = n_envs, a["num_agents"], obs_type, auto_reset
        self.tasks = tuple(int(m) for m in tasks) if tasks else None
        self.final_obs = bool(final_obs)
        if self.final_obs and not auto_reset:
            raise ValueError("final_obs needs auto_reset: without a reset no observation is overwritten")
        self.number_of_steps = kwargs.get("number_steps", 500)
        self.env_type = kwargs.get("env_type", 0)
        if self.env_type == 0 and self.number_of_steps < 1:
            raise ValueError("number_steps must be >= 1 for an episodic environment (env_type 0)")
        extra = {k: kwargs[k] for k in ("device", "rng_mode", "obs_dtype", "instance_base") if k in kwargs}
        self._env = BatchedGridEnvironment(n_envs, a["num_agents"], a["ticks_per_step"], a["arena_size"], a["pellet_regen"],
                                           a["num_pellets"], a["num_viruses"], a["num_bots"], a["reward_type"], a["c_death"],
                                           a["mode"], ram_obs=(2 if obs_type == "ram" else 0), tasks=self.tasks,
                                           pixel_obs=(int(pixel_size) if obs_type == "pixels" else 0), **extra)
        self._env.configure_observation({k: kwargs[k] for k in _OBS_KEYS if k in kwargs})
        self._ep_batch = None
        self._ep = None
        self._task = None
        self._start = None
        self._cell = None
        self._archive_select = False

    def seed(self, seed):
        self._env.seed(seed)

    def _obs(self):
        if self.obs_type == "grid":
            return self._env.batch.obs_tensor()
        if self.obs_type == "pixels":
            return self._env.batch.pixels()
        ram = self._env.ram()
        return ram[:, :self.num_agents, :]

    def reset(self):
        b = self._env.batch
        if self._ep_batch is not b:
            b.set_autoreset(self.number_of_steps if self.env_type == 0 else 0, self.final_obs, self.auto_reset)
            self._ep_batch = b
            self._ep = b.episode()
            final = {"grid": b.final_obs, "pixels": b.final_pixels}.get(self.obs_type, lambda: b.final_ram()[:, :self.num_agents, :])
            self._final = final() if self.final_obs else None
            self._task = b.tasks()["mode"] if self.tasks else None
        self._env.reset()  # (restarts every instance's step counter and return)
        return self._obs(), {}

    def step(self, dxdy, act):
        import torch
        assert self._ep is not None, "Cannot call step() before calling reset()"
        _, rew, _ = self._env.step_autoreset(dxdy, act)
        ep = self._ep
        done = ep["done"].view(torch.bool)
        info = {"steps": ep["steps"]}
        if self.auto_reset:
            info.update(reset_mask=ep["reset_mask"].view(torch.bool), episode_return=ep["episode_return"],
                        episode_length=ep["episode_length"])
            if self.final_obs:
                info["final_obs"] = self._final
        if self._task is not None:
            info["task"] = self._task
        if self._start is not None:
            info["start_result"] = self._start
        if self._cell is not None:
            info["cell"] = self._cell
        return self._obs(), rew.float(), done, torch.zeros_like(done), info

    def set_tasks(self, modes, number_steps=None):
        """what every environment plays from its next reset on: modes (int32 CUDA tensor of n_envs entries, -1 keeps the pending
        mode) and number_steps (int32 CUDA tensor or None: pending limits kept; -1 the constructor's number_steps, 0 none).
        Returns the per-environment result u8 [n_envs]: 0 nothing set, 1 set, 2 rejected (mode not in tasks, or limit < -1)"""
        if not self.tasks:
            raise ValueError("set_tasks needs a mixed-task environment (tasks=[...])")
        return self._env.set_tasks(modes, number_steps)

    def set_task_sizes(self, num_bots=None, num_pellets=None, num_viruses=None):
        """the game sizes every environment plays from its next reset on, each an int32 CUDA tensor of n_envs entries or None
        (pending values kept), -1 keeping an entry: num_bots (mode 0 only), num_pellets (not the squared-pellet modes 1, 2, 5)
        and num_viruses.  The constructor's counts are the maxima.  Returns the per-environment result u8 [n_envs]: 0 nothing
        set, 1 set, 2 rejected (a value above its maximum or below 0, or a bot count the player order does not allow)"""
        if not self.tasks:
            raise ValueError("set_task_sizes needs a mixed-task environment (tasks=[...])")
        return self._env.set_task_sizes(num_bots, num_pellets, num_viruses)

    # ---- snapshot pools (Batch.save_states / restore_states): save and restore whole games, episode counters included
    def snapshot_pool(self, slots):
        return self._env.snapshot_pool(slots)

    def save_states(self, pool, src, slots=None):
        """pool slot slots[k] (None: k) <- environment src[k] (int32 CUDA tensors), on the current stream"""
        assert self._ep is not None, "Cannot call save_states() before calling reset()"
        self._env.save_states(pool, src, slots)

    def restore_states(self, pool, slot_of):
        """environment i <- pool slot slot_of[i] where >= 0 (int32 CUDA tensor of n_envs entries); returns the observation.  A
        restored episode goes on counting towards number_steps from the step count it was saved with; restore_result() has the
        per-environment outcome (1 restored, 2 rejected)"""
        assert self._ep is not None, "Cannot call restore_states() before calling reset()"
        self._restore_result = self._env.restore_states(pool, slot_of)
        return self._obs()

    def set_start_states(self, pool, slot_of=None):
        """start states: from now on every reset of environment i with slot_of[i] >= 0 -- the auto-resets of step() and reset()
        -- begins the new episode in the game of pool slot slot_of[i] instead of a fresh spawn (int32 CUDA tensor of n_envs
        entries, -1: spawn; copied in stream order).  The new episode counts from 0 and continues the environment's own
        draw stream, so episodes started from one slot differ where the game draws.  info["start_result"] (u8 [n_envs]) then
        says how the last reset began: 0 not reset or spawned, 1 from its slot, 2 slot rejected and spawned.  pool None: every
        reset spawns again.  A Go-Explore loop keeps its archive on the device with set_archive, which chooses the slots itself:

            env.reset()
            env.set_archive(1024, cells_per_side=16)                          # 1024 cells, each with its best game
            for _ in range(steps):
                obs, rew, done, trunc, info = env.step(dxdy, act)             # finished episodes return into chosen cells
                bonus = env.archive()["visits"][info["cell"].clamp(min=0)]    # e.g. a count-based exploration bonus
        """
        self._env.set_start_states(pool, slot_of)
        self._start = self._env.batch.start_result() if pool is not None else None

    def set_archive(self, slots, cells_per_side=None, agent=0, select=True, seed=0):
        """attaches a Go-Explore cell archive of `slots` entries, in a pool of its own (snapshot_pool): every step() files each
        game under its cell -- agent `agent`'s position on a cells_per_side^2 grid and log2 of its mass -- and keeps the best
        game of every cell (highest trajectory score: the score of the cell the episode started from plus the episode's return,
        then the shortest trajectory).  With select, every reset -- the auto-resets of step() and reset() -- returns to a cell
        drawn with weight 1 / (1 + isqrt(times chosen)); info["start_result"] says which began in one.  info["cell"] (i32
        [n_envs], -1: no cell) is every environment's cell after the step.  Nothing is read back by the host.  slots None
        detaches it.  Call after reset(); archive() has the tables."""
        assert self._ep is not None, "Cannot call set_archive() before calling reset()"
        if slots is None:
            self._env.set_archive(None)
            self._cell = None
            if self._archive_select:
                self._start = None
            self._archive_select = False
            return
        self._env.set_archive(self._env.snapshot_pool(slots), cells_per_side, agent, select, seed)
        self._cell = self._env.archive()["cell_of"]
        if select:
            self._start = self._env.batch.start_result()
        elif self._archive_select:
            self._start = None
        self._archive_select = bool(select)

    def archive(self):
        """device views of the archive (Batch.archive): cell_of, base_score, base_length, key_entry, visits, entry_key,
        entry_score, entry_length, entry_chosen, counters (used, dropped, improved)"""
        return self._env.archive()

    def restore_result(self):
        """u8 [n_envs] of the last restore_states: 0 not requested, 1 restored, 2 rejected"""
        return self._restore_result

    def flags(self):
        """(OR over all instances, {AGARCL_FLAG name: instances}) -- fixed capacities hit since the instances' last reset"""
        return self._env.flags()

    def bot_actions(self, types, out=None):
        """what a built-in bot (BOT_HUNGRY .. BOT_AGGRESSIVE_SHY, agarcl_b200.BOT_TYPES) would do for every agent on the current
        games: (dxdy f32 [n_envs * num_agents, 2], act i32, status u8) device tensors on the current stream, without a host wait.
        dxdy and act go straight into step(): a scripted baseline, expert actions for imitation, or scripted partners and
        opponents.  types: one type for every agent, or an int32 CUDA tensor with -1 for the agents a learner drives (their
        entries are left as they are, so `out` can be an action buffer the policy already filled).  dxdy is not clamped to the
        action box: the step moves towards the target the bot chose.  status: 1 decided, 2 no pellet left (dxdy 0), 3 the agent
        is dead (dxdy 0), 0 skipped, 4 not a bot type"""
        return self._env.bot_actions(types, out)

    def render(self, env_ids=None, size=256, view="arena", out=None):
        """RGB pictures uint8 [n, size, size, 3] (device tensor) of the current games, drawn on the device on the current torch
        stream without a host wait (Batch.draw).  env_ids: int32 CUDA tensor of environments, or None for all.  view "arena": one
        picture per environment; "agent": one per agent, environment-major (n * num_agents pictures), each the window of that
        agent's grid observation.  out: a preallocated uint8 CUDA tensor of that shape, e.g. a slice of a video buffer."""
        import torch
        b = self._env.batch
        src = env_ids.to(torch.int32) if env_ids is not None else None
        if view == "agent" and src is not None:
            A = self.num_agents
            src = (src.view(-1, 1) * A + torch.arange(A, dtype=torch.int32, device=src.device)).view(-1)
        return b.draw(src, size, view, out)  # (the stream the steps run on)

    def close(self):
        self._env.close()


_REGISTRY = {"agario-grid-v0": "grid", "agario-gobigger-v0": "gobigger", "agario-ram-v0": "ram"}


def make(env_id, **kwargs):
    """gym.make for the ids gym_agario registers (gym_agario/__init__.py:9-23)"""
    if env_id not in _REGISTRY:
        raise ValueError(f"unknown environment id {env_id}")
    return AgarioEnv(obs_type=_REGISTRY[env_id], **kwargs)


if gym is not None:  # pragma: no cover
    from gymnasium.envs.registration import register, registry
    for _id, _t in _REGISTRY.items():
        if _id not in registry:
            register(id=_id, entry_point="agarcl_b200.gym_env:AgarioEnv", kwargs={"obs_type": _t})
