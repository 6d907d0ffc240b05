"""Shared test plumbing: loads the checkers (oracle port, compiled reference, picture and bot oracles) and the product
library through ctypes and offers small wrappers.  TEST INFRASTRUCTURE ONLY."""
import atexit
import ctypes as C
import hashlib
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np

from agarcl_b200._abi import (BOT_DEAD, BOT_DECIDED, BOT_NO_PELLET, Cfg, Layout, RAM_RECORD, StateView, compare_states, make_cfg)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libagarcl_ref.so")
PRODUCT_SO = os.path.join(ROOT, "agarcl_b200", "libagarcl_b200.so")
NO_REF = "compiled reference not available: set AGARCL_REFERENCE to an AgarCL checkout to build it"
LIBSTDCXX_GOLDEN = os.path.join(ROOT, "tests", "golden", "libstdcxx")


def inputs_digest(inputs):
    h = hashlib.sha256()
    for a in inputs:
        a = np.ascontiguousarray(a)
        h.update(np.int64(a.size).tobytes() + a.dtype.str.encode() + a.tobytes())
    return h.hexdigest()


def libstdcxx_expected(name, inputs):
    """What libstdc++ itself returned for each of `inputs` (tests/golden/libstdcxx/<name>.npz, written by
    tests/golden/make_libstdcxx_golden.py with the code of oracle/ref_harness.cpp), one int32 array per input."""
    z = np.load(os.path.join(LIBSTDCXX_GOLDEN, name + ".npz"))
    assert str(z["inputs_sha256"]) == inputs_digest(inputs), \
        f"{name}: the seeded inputs changed, regenerate with python tests/golden/make_libstdcxx_golden.py"
    return np.split(z["out"].astype(np.int32), np.cumsum([np.size(a) for a in inputs])[:-1])


_vp = C.c_void_p


def fptr(a):
    return a.ctypes.data_as(_vp)


def _build():
    if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(os.path.join(ROOT, "oracle", "oracle.c")):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"], stdout=subprocess.DEVNULL)
    if not os.path.exists(REF_SO) and os.environ.get("AGARCL_REFERENCE"):  # (make fails when it names no AgarCL tree)
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref"], stdout=subprocess.DEVNULL)


_oracle = None
_ref = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        _build()
        _oracle = C.CDLL(ORACLE_SO)
        _oracle.oracle_make_layout.restype = C.c_int
    return _oracle


def ref_lib():
    """The compiled reference engine, or None when it has not been built (AGARCL_REFERENCE not set)."""
    global _ref
    if _ref is None:
        _build()
        if not os.path.exists(REF_SO):
            return None
        _ref = C.CDLL(REF_SO)
        _ref.ref_create.restype = _vp
        _ref.ref_bench.restype = C.c_double
    return _ref


def oracle_layout(cfg):
    L = Layout()
    rc = oracle_lib().oracle_make_layout(C.byref(cfg), C.byref(L))
    assert rc == 0, "oracle_make_layout failed"
    return L


class Oracle:
    """One instance stepped by oracle/oracle.c."""

    def __init__(self, cfg, layout=None, replay=None):
        self.lib = oracle_lib()
        self.cfg = cfg
        self.L = layout or oracle_layout(cfg)
        self.state = StateView(self.L)
        self.replay = np.ascontiguousarray(replay if replay is not None else np.zeros(0, np.float32), dtype=np.float32)

    def set_replay(self, replay):
        self.replay = np.ascontiguousarray(replay, dtype=np.float32)

    def seed_mt(self, seed, n=1 << 16):
        d = np.zeros(n, np.float32)
        self.lib.oracle_mt19937_draws(C.c_uint64(seed), fptr(d), n)
        self.replay = d

    def reset(self):
        self.lib.oracle_reset(C.byref(self.cfg), C.byref(self.L), self.state.ptr, fptr(self.replay), self.replay.size)

    def reset_keep_stream(self):
        """a later episode: the draw stream goes on (Engine::reset does not reseed)"""
        self.lib.oracle_reset_keep_stream(C.byref(self.cfg), C.byref(self.L), self.state.ptr, fptr(self.replay), self.replay.size)

    def set_actions(self, dxdy, act):
        dxdy = np.ascontiguousarray(dxdy, np.float32)
        act = np.ascontiguousarray(act, np.int32)
        self.lib.oracle_set_actions(C.byref(self.cfg), C.byref(self.L), self.state.ptr, fptr(dxdy), fptr(act))

    def step(self, with_obs=False):
        A = self.L.A
        rew = np.zeros(A, np.float64)
        dones = np.zeros(A, np.uint8)
        obs = None
        if with_obs:
            obs = np.zeros((A, self.cfg.num_frames * self.L.obs_channels, self.cfg.grid_size, self.cfg.grid_size), np.int32)
        self.lib.oracle_step(C.byref(self.cfg), C.byref(self.L), self.state.ptr, fptr(self.replay), self.replay.size,
                             fptr(rew), fptr(dones), fptr(obs) if with_obs else None)
        return rew, dones, obs

    def obs(self, agent):
        out = np.zeros((self.L.obs_channels, self.cfg.grid_size, self.cfg.grid_size), np.int32)
        self.lib.oracle_obs(C.byref(self.cfg), C.byref(self.L), self.state.ptr, agent, 0, fptr(out))
        return out

    # ---- structured ("ram") observation: records persist between calls (players with nothing in view keep theirs)
    def ram_clear(self):
        self.ram = np.zeros((self.L.P, RAM_RECORD), np.float32)

    def ram_obs(self):
        """oracle_ram_obs on the CURRENT state"""
        if not hasattr(self, "ram"):
            self.ram_clear()
        self.lib.oracle_ram_obs(C.byref(self.cfg), C.byref(self.L), self.state.ptr, fptr(self.ram))
        return self.ram

    def step_with_ram(self, with_obs=False):
        """oracle_step with the records taken where the reference takes them (after the ticks, before respawn)"""
        if not hasattr(self, "ram"):
            self.ram_clear()
        self.lib.oracle_set_ram_out(fptr(self.ram))
        try:
            return self.step(with_obs=with_obs)
        finally:
            self.lib.oracle_set_ram_out(None)


def aged_oracle(kw, seed, steps, boost=None):
    """an oracle of make_cfg(**kw) on the mt19937 stream of `seed`, reset (the agents' first cell at mass `boost`, when given)
    and stepped `steps` times with random actions (p_feed = p_split = 0.3)"""
    oracle_lib().oracle_set_trig_mode(1)
    cfg = make_cfg(rng_mode=1, cap_replay=1 << 16, **kw)
    o = Oracle(cfg)
    o.seed_mt(seed)
    o.reset()
    if boost:
        for a in range(o.L.A):
            o.state.cells[a][0]["mass"] = boost
    rng = np.random.default_rng(seed)
    for _ in range(steps):
        o.set_actions(*random_actions(rng, o.L.A, 0.3, 0.3))
        o.step()
    return o


def _compile_once(name, extra_flags=()):
    """tests/<name>.c compiled once per session into a temporary directory (the tree may be read-only)"""
    d = tempfile.mkdtemp(prefix=f"agarcl_{name}_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, f"lib{name}.so")
    subprocess.check_call(["gcc", "-std=c11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wall", *extra_flags,
                           "-o", so, os.path.join(ROOT, "tests", f"{name}.c"), "-lm"])
    return C.CDLL(so)


# ---- pictures of game states: tests/draw_oracle.c
ARENA, AGENT = 0, 1


def _rgb_constants():
    """AGARCL_DRAW_RGB_* of the header, as (r, g, b) tuples (the palettes as lists of them)"""
    text = open(os.path.join(ROOT, "include", "agarcl_b200.h")).read()
    rgb = lambda v: ((v >> 16) & 255, (v >> 8) & 255, v & 255)  # noqa: E731
    out = {m.group(1): rgb(int(m.group(2), 16)) for m in re.finditer(r"#define AGARCL_DRAW_RGB_(\w+) (0x[0-9A-Fa-f]+)u", text)}
    for name in ("AGENTS", "BOTS"):
        body = re.search(r"#define AGARCL_DRAW_RGB_%s \{([^}]*)\}" % name, text).group(1)
        out[name] = [rgb(int(v.strip().rstrip("u"), 16)) for v in body.split(",")]
    return out


RGB = _rgb_constants()
_draw_lib = None


def oracle_draw(cfg, L, blob, view, agent, size):
    global _draw_lib
    if _draw_lib is None:
        _draw_lib = _compile_once("draw_oracle")
    out = np.zeros((size, size, 3), np.uint8)
    _draw_lib.oracle_draw(C.byref(cfg), C.byref(L), blob.ctypes.data_as(C.c_void_p), int(view), int(agent), int(size),
                          out.ctypes.data_as(C.c_void_p))
    return out


# ---- built-in bot policies: tests/bot_oracle.c (which includes oracle/oracle.c, compiled with the oracle's flags)
_bot_lib = None


def oracle_bot_decide(cfg, L, blob, agent, bot_type):
    """(dxdy f32 [2], target f32 [2], act, status) of oracle_bot_decide"""
    global _bot_lib
    if _bot_lib is None:
        _bot_lib = _compile_once("bot_oracle", ["-Wno-unused-function"])
    dxdy, target = np.zeros(2, np.float32), np.zeros(2, np.float32)
    act, status = C.c_int32(0), C.c_uint8(0)
    vp = C.c_void_p
    _bot_lib.oracle_bot_decide(C.byref(cfg), C.byref(L), blob.ctypes.data_as(vp), int(agent), int(bot_type),
                               dxdy.ctypes.data_as(vp), target.ctypes.data_as(vp), C.byref(act), C.byref(status))
    return dxdy, target, int(act.value), int(status.value)


def oracle_bot_batch(cfg, L, blobs, types):
    """every agent of the blobs [N][stride] with types [N*A]: dxdy [N*A, 2], target [N*A, 2], act [N*A], status [N*A]; skipped
    and bad-type agents are left at 0"""
    NA = len(blobs) * L.A
    dxdy, target = np.zeros((NA, 2), np.float32), np.zeros((NA, 2), np.float32)
    act, status = np.zeros(NA, np.int32), np.zeros(NA, np.uint8)
    for j in range(NA):
        d, t, a, s = oracle_bot_decide(cfg, L, blobs[j // L.A], j % L.A, int(types[j]))
        status[j] = s
        if s in (BOT_DECIDED, BOT_NO_PELLET, BOT_DEAD):
            dxdy[j], target[j], act[j] = d, t, a
    return dxdy, target, act, status


class Reference:
    """One instance of the compiled reference GridEnvironment<int,false>."""

    def __init__(self, cfg, layout):
        self.lib = ref_lib()
        assert self.lib is not None
        self.cfg, self.L = cfg, layout
        self.h = _vp(self.lib.ref_create(C.byref(cfg)))

    def __del__(self):
        try:
            self.lib.ref_destroy(self.h)
        except Exception:
            pass

    def seed(self, s):
        self.lib.ref_seed(self.h, C.c_uint(s))

    def reset(self):
        self.lib.ref_reset(self.h)

    def reset_native(self):
        """BaseEnvironment::reset as the reference runs it (pids keep counting, quirk Q3)"""
        self.lib.ref_reset_native(self.h)

    def pid_base(self):
        return int(self.lib.ref_pid_base(self.h))

    def order(self):
        o = (C.c_int32 * 64)()
        n = self.lib.ref_player_order(self.h, o)
        return list(o)[:n]

    def peek_draws(self, n):
        d = np.zeros(n, np.float32)
        self.lib.ref_rng_peek(self.h, fptr(d), n)
        return d

    def dump(self):
        sv = StateView(self.L)
        miss = self.lib.ref_dump_state(self.h, C.byref(self.L), sv.ptr)
        return sv, miss

    def set_actions(self, dxdy, act):
        dxdy = np.ascontiguousarray(dxdy, np.float32)
        act = np.ascontiguousarray(act, np.int32)
        self.lib.ref_take_actions(self.h, fptr(dxdy), fptr(act))

    def step(self):
        """rewards re-indexed by agent (the reference returns them in player-map order, quirk Q15)"""
        A = self.L.A
        raw = np.zeros(A, np.float64)
        self.lib.ref_step(self.h, fptr(raw))
        agents_in_map_order = [p for p in self.order() if p < A]
        rew = np.zeros(A, np.float64)
        for j, p in enumerate(agents_in_map_order):
            rew[p] = raw[j]
        d = np.zeros(A, np.uint8)
        self.lib.ref_dones(self.h, fptr(d))
        return rew, d

    def obs(self, agent):
        out = np.zeros((self.L.obs_channels, self.cfg.grid_size, self.cfg.grid_size), np.int32)
        self.lib.ref_obs(self.h, agent, fptr(out))
        return out

    def ram_clear(self):
        self.ram = np.zeros((self.L.P, RAM_RECORD), np.float32)
        self.lib.ref_ram_clear(self.h)

    def ram_obs(self):
        """GoBiggerObservation::add_frame on the current reference state, flattened into agarcl records"""
        if not hasattr(self, "ram"):
            self.ram_clear()
        self.lib.ref_ram_obs(self.h, self.L.P, fptr(self.ram))
        return self.ram

    def agent_pids(self):
        o = (C.c_int32 * 64)()
        n = self.lib.ref_agent_pids(self.h, o)
        return list(o)[:n]

    def save_env_state(self, path):
        assert self.lib.ref_save_env_state(self.h, str(path).encode()) == 0

    def load_env_state(self, path):
        assert self.lib.ref_load_env_state(self.h, str(path).encode()) == 0

    def set_cell_mass(self, pid, cell, mass):
        self.lib.ref_set_cell_mass(self.h, pid, cell, C.c_uint(mass))

    def set_cell_pos(self, pid, cell, x, y):
        self.lib.ref_set_cell_pos(self.h, pid, cell, C.c_float(x), C.c_float(y))

    def set_virus(self, idx, x, y):
        self.lib.ref_set_virus(self.h, idx, C.c_float(x), C.c_float(y))


def random_actions(rng, A, p_feed=1 / 3, p_split=1 / 3):
    dxdy = rng.uniform(-1, 1, size=(A, 2)).astype(np.float32)
    u = rng.random(A)
    act = np.where(u < p_feed, 1, np.where(u < p_feed + p_split, 2, 0)).astype(np.int32)
    return dxdy, act
