"""Batch handle: thin Python owner of an `agarcl_batch*` (include/agarcl_b200.h).

This is the host-side mirror of the batched hot path.  Device buffers are owned by the C library;
`obs_tensor()/rewards_tensor()/dones_tensor()` expose them to PyTorch without a copy through
`__cuda_array_interface__` (torch is plumbing here: device memory views and streams only).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._abi import DRAW_VIEWS, FLAG_NAMES, OBS_I16, RAM_RECORD, Archive, ArchiveCfg, Layout, StateView

_vp = C.c_void_p


class _CudaView:
    def __init__(self, ptr, shape, typestr, owner):
        self.__cuda_array_interface__ = {"shape": tuple(int(s) for s in shape), "typestr": typestr,
                                         "data": (int(ptr), False), "version": 2}
        self._owner = owner


class _ObsListsStruct(C.Structure):
    """struct agarcl_obs_lists"""
    _fields_ = [(n, C.c_int32) for n in ("n_images", "n_chunks", "images_per_chunk", "frames", "channels", "grid", "obs_dtype",
                                         "mask_words", "rec_words", "entries_per_image")] + \
               [(n, C.c_uint32) for n in ("off_rec", "off_entries", "chunk_words")] + [("chunks", _vp), ("slot_of", _vp)]


class _EpisodeStruct(C.Structure):
    """struct agarcl_episode"""
    _fields_ = [(n, _vp) for n in ("done_out", "reset_mask", "steps", "final_return", "final_length", "final_obs", "final_ram")]


class _TasksStruct(C.Structure):
    """struct agarcl_tasks"""
    _fields_ = [(n, _vp) for n in ("mode", "max_steps", "next_mode", "next_max_steps")]


class _TaskSizesStruct(C.Structure):
    """struct agarcl_task_sizes"""
    _fields_ = [(n, _vp) for n in ("bots", "pellets", "viruses", "next_bots", "next_pellets", "next_viruses")]


class ObsLists:
    """numpy view of the lists of the last Batch.step_lists (layout: include/agarcl_b200.h, agarcl_obs_lists)"""

    def __init__(self, batch, L):
        self._b, self.L = batch, L
        words = L.n_chunks * L.chunk_words
        self.words = np.ctypeslib.as_array(C.cast(L.chunks, C.POINTER(C.c_uint32)), shape=(words,))
        self.slot_of = np.ctypeslib.as_array(C.cast(L.slot_of, C.POINTER(C.c_uint32)), shape=(L.n_images,))

    def record(self, image):
        L = self.L
        s = int(self.slot_of[image])
        c, li = divmod(s, L.images_per_chunk)
        base = c * L.chunk_words
        rec = self.words[base + L.off_rec + li * L.rec_words: base + L.off_rec + (li + 1) * L.rec_words]
        return c, rec

    def entries(self, image):
        """(op, element offset, operand) arrays of the image, in application order; None if it overflowed its slot"""
        L = self.L
        c, rec = self.record(image)
        if int(rec[0]) == 0xFFFFFFFF:
            return None
        e0 = c * L.chunk_words + L.off_entries + 2 * int(rec[1])
        e = self.words[e0: e0 + 2 * int(rec[0])].reshape(-1, 2)
        return e[:, 0] >> 29, e[:, 0] & 0x1FFFFFFF, e[:, 1].astype(np.int64)

    def decode(self, image):
        """pure-numpy decoder of one image from the documented layout (what a consumer writes; the C decoder is expand())"""
        L = self.L
        G, CH = L.grid, L.frames * L.channels
        dt = np.int16 if L.obs_dtype == OBS_I16 else np.int32
        top = 32767 if dt == np.int16 else 2147483647
        out = np.zeros((CH, G, G), np.int64)
        _, rec = self.record(image)
        ent = self.entries(image)
        if ent is None:
            return None
        for f in range(L.frames):
            m = rec[3 + 2 * f * L.mask_words: 3 + 2 * (f + 1) * L.mask_words]
            bits = lambda w: np.unpackbits(w.view(np.uint8), bitorder="little")[:G].astype(bool)  # noqa: E731
            rows, cols = bits(m[:L.mask_words].copy()), bits(m[L.mask_words:].copy())
            out[f * L.channels][rows[:, None] | cols[None, :]] = -1
        flat = out.reshape(-1)
        for op, off, v in zip(*ent):
            x = flat[off]
            v = min(int(v), top)
            flat[off] = v if op == 0 else min(x + v, top) if op == 1 else (x if (x != 0 and x < v) else v) if op == 2 else max(x, v)
        return out.astype(dt)

    def expand(self, image):
        """dense [frames*C, G, G] frame of one image (C decoder, agarcl_batch_lists_expand)"""
        L = self.L
        out = np.empty((L.frames * L.channels, L.grid, L.grid), np.int16 if L.obs_dtype == OBS_I16 else np.int32)
        _lib.check(_lib.lib().agarcl_batch_lists_expand(self._b._h, int(image), out.ctypes.data_as(_vp)))
        return out

    def rewards_dones(self):
        """(rewards f64 [n_images], dones u8 [n_images]) read from the records"""
        L = self.L
        rew, done = np.zeros(L.n_images, np.float64), np.zeros(L.n_images, np.uint8)
        for i in range(L.n_images):
            _, rec = self.record(i)
            rew[i] = rec[L.rec_words - 3: L.rec_words - 1].copy().view(np.float64)[0]
            done[i] = rec[L.rec_words - 1]
        return rew, done


class Batch:
    def __init__(self, cfg):
        self.cfg = cfg
        self._h = _vp()
        _lib.check(_lib.lib().agarcl_batch_create(C.byref(cfg), C.byref(self._h)))
        self.layout = Layout()
        _lib.check(_lib.lib().agarcl_batch_get_layout(self._h, C.byref(self.layout)))
        self.N = cfg.n_instances
        self.A = self.layout.A
        shape = (C.c_int64 * 4)()
        ptr = _vp()
        dt = C.c_int32()
        _lib.check(_lib.lib().agarcl_batch_obs(self._h, C.byref(ptr), C.byref(shape), C.byref(dt)))
        self.obs_shape = tuple(int(x) for x in shape)
        self.obs_dtype = np.int16 if dt.value == OBS_I16 else np.int32
        self._obs_ptr = ptr.value
        p = _vp()
        _lib.check(_lib.lib().agarcl_batch_rewards(self._h, C.byref(p)))
        self._rew_ptr = p.value
        p = _vp()
        _lib.check(_lib.lib().agarcl_batch_dones(self._h, C.byref(p)))
        self._done_ptr = p.value

    def close(self):
        if self._h:
            self._mirror = None
            _lib.lib().agarcl_batch_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def _device(self):
        return torch.device("cuda", self.cfg.device)

    def _tensor(self, ptr, shape, typestr):
        """zero-copy torch view of library-owned device memory (typestr: numpy's, "<f4"); it keeps the batch alive"""
        return torch.as_tensor(_CudaView(ptr, shape, typestr, self), device=self._device)

    # ---- reference-shaped calls
    def seed(self, seeds):
        s = np.ascontiguousarray(np.broadcast_to(np.asarray(seeds, dtype=np.uint64), (self.N,)) if np.ndim(seeds) else
                                 np.arange(self.N, dtype=np.uint64) + np.uint64(seeds))
        _lib.check(_lib.lib().agarcl_batch_seed(self._h, s.ctypes.data_as(_vp)))

    def reset(self, mask=None, stream=0):
        m = None
        if mask is not None:
            m = np.ascontiguousarray(mask, dtype=np.uint8)
            if m.size != self.N:
                raise _lib.AgarclError(f"the reset mask must have {self.N} entries (one per instance), got {m.size}")
        _lib.check(_lib.lib().agarcl_batch_reset(self._h, m.ctypes.data_as(_vp) if m is not None else None, _vp(stream)))
        if m is None:  # strict_reference: the player order of the new episode (quirk Q3)
            _lib.check(_lib.lib().agarcl_batch_get_layout(self._h, C.byref(self.layout)))

    def reset_device(self, mask, stream=0):
        """masked reset with a CUDA uint8 / bool tensor of N entries: read by the device, the host does not wait"""
        self._check_device_tensor(mask, (torch.uint8, torch.bool), "the reset mask", self.N)
        _lib.check(_lib.lib().agarcl_batch_reset_device(self._h, _vp(mask.data_ptr()), _vp(stream)))

    def set_autoreset(self, max_steps=0, keep_final_obs=False, reset=True):
        """enables the episode bookkeeping of step_autoreset (include/agarcl_b200.h, agarcl_batch_set_autoreset)"""
        _lib.check(_lib.lib().agarcl_batch_set_autoreset(self._h, int(max_steps), int(bool(keep_final_obs)), int(bool(reset))))
        self._episode = None

    def step_autoreset(self, stream=0):
        """step, then on the device: done flags with the step limit, the reset mask, episode statistics, the final observation
        (when kept) and the reset of the finished instances"""
        _lib.check(_lib.lib().agarcl_batch_step_autoreset(self._h, _vp(stream)))

    def _episode_struct(self):
        if getattr(self, "_episode", None) is None:
            e = _EpisodeStruct()
            _lib.check(_lib.lib().agarcl_batch_episode(self._h, C.byref(e)))
            self._episode = e
        return self._episode

    def episode(self):
        """zero-copy device views of the episode buffers, overwritten by every step_autoreset: done (u8 [N*A]), reset_mask
        (u8 [N]), steps (i64 [N]), episode_return (f64 [N*A]) and episode_length (i64 [N]); the last two hold each instance's
        last finished episode, to be read where reset_mask is set"""
        e, N, NA = self._episode_struct(), self.N, self.N * self.A
        return {"done": self._tensor(e.done_out, (NA,), "|u1"), "reset_mask": self._tensor(e.reset_mask, (N,), "|u1"),
                "steps": self._tensor(e.steps, (N,), "<i8"), "episode_return": self._tensor(e.final_return, (NA,), "<f8"),
                "episode_length": self._tensor(e.final_length, (N,), "<i8")}

    def final_obs(self):
        """observation images [N*A, frames*C, G, G] the reset instances of the last step_autoreset ended their episode on"""
        e = self._episode_struct()
        if not e.final_obs:
            raise _lib.AgarclError("no final observation images: set_autoreset(keep_final_obs=True) with a grid observation")
        return self._tensor(e.final_obs, self.obs_shape, np.dtype(self.obs_dtype).str)

    def final_ram(self):
        """ram records [N, P, RAM_RECORD] float32 the reset instances of the last step_autoreset ended their episode on"""
        e = self._episode_struct()
        if not e.final_ram:
            raise _lib.AgarclError("no final ram records: set_autoreset(keep_final_obs=True) with cfg.ram_obs")
        return self._tensor(e.final_ram, (self.N, self.layout.P, RAM_RECORD), "<f4")

    def set_actions(self, dxdy, act, stream=0):
        """the actions of the next step: dxdy [N*A, 2] float32 and act [N*A] int32, as host arrays (converted and copied) or as
        CUDA tensors on the batch's device (read by the device in place, so they are not converted: another dtype is refused)"""
        if isinstance(dxdy, torch.Tensor) or isinstance(act, torch.Tensor):
            self._check_device_tensor(dxdy, torch.float32, "dxdy")
            self._check_device_tensor(act, torch.int32, "act")
            self._check_action_sizes(dxdy.numel(), act.numel())
            self.set_actions_device(dxdy.data_ptr(), act.data_ptr(), stream)
            return
        dxdy, act = self._host_actions(dxdy, act)
        _lib.check(_lib.lib().agarcl_batch_set_actions(self._h, dxdy.ctypes.data_as(_vp), act.ctypes.data_as(_vp), 0, _vp(stream)))

    def set_actions_device(self, dxdy_ptr, act_ptr, stream=0):
        _lib.check(_lib.lib().agarcl_batch_set_actions(self._h, _vp(dxdy_ptr), _vp(act_ptr), 1, _vp(stream)))

    def step(self, stream=0):
        _lib.check(_lib.lib().agarcl_batch_step(self._h, _vp(stream)))

    def render(self, stream=0):
        _lib.check(_lib.lib().agarcl_batch_render(self._h, _vp(stream)))

    def render_ram(self, stream=0):
        _lib.check(_lib.lib().agarcl_batch_render_ram(self._h, _vp(stream)))

    def ram_tensor(self):
        """structured observation records [N, P, RAM_RECORD] float32 on the device (cfg.ram_obs)"""
        p, shape = _vp(), (C.c_int64 * 3)()
        _lib.check(_lib.lib().agarcl_batch_ram(self._h, C.byref(p), C.byref(shape)))
        return self._tensor(p.value, tuple(shape), "<f4")

    def _check_action_sizes(self, n_dxdy, n_act):
        """the C ABI reads N*A (dx, dy) float32 pairs and N*A int32 actions"""
        if n_dxdy != self.N * self.A * 2 or n_act != self.N * self.A:
            raise _lib.AgarclError(f"Number of actions does not match number of agents ({self.N * self.A})")

    def _host_actions(self, dxdy, act):
        """the C ABI reads raw float32 / int32 buffers: coerce (and check the sizes of) whatever the caller hands in"""
        dxdy = np.ascontiguousarray(dxdy, dtype=np.float32)
        act = np.ascontiguousarray(act, dtype=np.int32)
        self._check_action_sizes(dxdy.size, act.size)
        return dxdy, act

    @staticmethod
    def _host_out(a, dtype, size, what):
        if a is None:
            return None
        if not (isinstance(a, np.ndarray) and a.dtype == dtype and a.flags.c_contiguous and a.size == size):
            raise _lib.AgarclError(f"{what} must be a C-contiguous {np.dtype(dtype).name} array of {size} elements")
        return a.ctypes.data_as(_vp)

    def step_host(self, dxdy, act, obs_out=None, rewards_out=None, dones_out=None):
        dxdy, act = self._host_actions(dxdy, act)
        NA = self.N * self.A
        _lib.check(_lib.lib().agarcl_batch_step_host(
            self._h, dxdy.ctypes.data_as(_vp), act.ctypes.data_as(_vp),
            self._host_out(obs_out, self.obs_dtype, int(np.prod(self.obs_shape)), "obs_out"),
            self._host_out(rewards_out, np.float64, NA, "rewards_out"), self._host_out(dones_out, np.uint8, NA, "dones_out")))

    # ---- host-resident observation mirror (include/agarcl_b200.h, mirror.cu)
    def mirror(self):
        """numpy view [N*A, C*frames, G, G] of the library-owned pinned host mirror of the observation (read-only)"""
        if getattr(self, "_mirror", None) is None:
            p, shape, dt = _vp(), (C.c_int64 * 4)(), C.c_int32()
            _lib.check(_lib.lib().agarcl_batch_mirror(self._h, C.byref(p), C.byref(shape), C.byref(dt)))
            n = int(np.prod(list(shape)))
            ct = C.c_int16 if dt.value == OBS_I16 else C.c_int32
            a = np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), shape=(n,)).reshape(tuple(int(x) for x in shape))
            a.flags.writeable = False
            self._mirror = a
        return self._mirror

    def sync_mirror(self, stream=0):
        self.mirror()
        _lib.check(_lib.lib().agarcl_batch_sync_mirror(self._h, _vp(stream)))
        return self._mirror

    def step_mirror(self, dxdy, act, rewards_out=None, dones_out=None):
        """take_actions (host arrays) + step + mirror sync; returns the mirror view"""
        dxdy, act = self._host_actions(dxdy, act)
        NA = self.N * self.A
        self.mirror()
        _lib.check(_lib.lib().agarcl_batch_step_mirror(
            self._h, dxdy.ctypes.data_as(_vp), act.ctypes.data_as(_vp),
            self._host_out(rewards_out, np.float64, NA, "rewards_out"), self._host_out(dones_out, np.uint8, NA, "dones_out")))
        return self._mirror

    # ---- the observation as lists (include/agarcl_b200.h, agarcl_obs_lists): no dense host tensor, nothing to patch
    def step_lists(self, dxdy, act, rewards_out=None, dones_out=None):
        """take_actions (host arrays) + step; rewards / dones to host; returns an ObsLists view of the library-owned pinned
        lists (valid until the next step call)"""
        dxdy, act = self._host_actions(dxdy, act)
        NA = self.N * self.A
        L = _ObsListsStruct()
        _lib.check(_lib.lib().agarcl_batch_step_lists(
            self._h, dxdy.ctypes.data_as(_vp), act.ctypes.data_as(_vp),
            self._host_out(rewards_out, np.float64, NA, "rewards_out"), self._host_out(dones_out, np.uint8, NA, "dones_out"), C.byref(L)))
        return ObsLists(self, L)

    def mirror_stats(self):
        out = (C.c_uint64 * 4)()
        _lib.check(_lib.lib().agarcl_batch_mirror_stats(self._h, C.byref(out)))
        t = (C.c_uint64 * 4)()
        _lib.check(_lib.lib().agarcl_batch_mirror_timing(self._h, C.byref(t)))
        return dict(entries=int(out[0]), dense_images=int(out[1]), d2h_bytes=int(out[2]), host_threads=int(out[3]),
                    wait_us=int(t[0]), total_us=int(t[1]), launch_us=int(t[2]), call_us=int(t[3]))

    def set_timing(self, enable=True):
        _lib.check(_lib.lib().agarcl_batch_set_timing(self._h, int(enable)))

    def get_timing(self):
        """(engine-tick kernel ms, observation kernel ms, steps) accumulated since the last call"""
        a, o, n = C.c_double(), C.c_double(), C.c_int32()
        _lib.check(_lib.lib().agarcl_batch_get_timing(self._h, C.byref(a), C.byref(o), C.byref(n)))
        return a.value, o.value, n.value

    def launches_per_step(self):
        return _lib.lib().agarcl_batch_launches_per_step(self._h)

    def flags(self, stream=0):
        """(OR of hdr.flags over all instances, {flag name: instances with it set}); reduced on the device"""
        o, counts = C.c_uint32(), (C.c_uint32 * 32)()
        _lib.check(_lib.lib().agarcl_batch_flags(self._h, _vp(stream), C.byref(o), C.byref(counts)))
        return int(o.value), {FLAG_NAMES.get(1 << i, f"bit{i}"): int(counts[i]) for i in range(32) if counts[i]}

    # ---- snapshot pools (include/agarcl_b200.h, agarcl_batch_save_states / agarcl_batch_restore_states)
    @property
    def slot_bytes(self):
        """bytes of one snapshot slot of this batch's configuration"""
        if getattr(self, "_slot_bytes", None) is None:
            self._slot_bytes = _lib.snapshot_slot_bytes(self.cfg)
        return self._slot_bytes

    def snapshot_pool(self, slots):
        """a zeroed pool of `slots` slots: torch.uint8 [slots, slot_bytes] on the batch's device"""
        if int(slots) < 1:
            raise _lib.AgarclError("a pool needs at least one slot")
        return torch.zeros((int(slots), self.slot_bytes), dtype=torch.uint8, device=self._device)

    def _check_device_tensor(self, t, dtype, what, numel=None):
        """refuses what the library could not read as `what`: dtype is a torch dtype or a tuple of those allowed"""
        dtypes = dtype if isinstance(dtype, tuple) else (dtype,)
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.device == self._device):
            raise _lib.AgarclError(f"{what} must be a tensor on {self._device}")
        if t.dtype not in dtypes:
            raise _lib.AgarclError(f"{what} must be {' or '.join(str(d).removeprefix('torch.') for d in dtypes)}, got {t.dtype}")
        if not t.is_contiguous():
            raise _lib.AgarclError(f"{what} must be contiguous" + (f" with {numel} entries" if numel is not None else ""))
        if numel is not None and t.numel() != numel:
            raise _lib.AgarclError(f"{what} must have {numel} entries, got {t.numel()}")

    def _check_pool(self, pool):
        self._check_device_tensor(pool, torch.uint8, "the pool")
        if pool.dim() != 2 or pool.shape[1] != self.slot_bytes or pool.shape[0] < 1:
            raise _lib.AgarclError(f"the pool must be [slots >= 1, {self.slot_bytes}] (slot bytes of this configuration), "
                                   f"got {list(pool.shape)}")
        return int(pool.shape[0])

    def save_states(self, pool, src, slots=None, stream=0):
        """pool slot slots[k] (None: slot k) <- instance src[k], for every k; int32 CUDA tensors; enqueued on `stream`, no host
        wait.  A slot index out of range is skipped; a source out of range leaves a slot that restores reject."""
        n_slots = self._check_pool(pool)
        self._check_device_tensor(src, torch.int32, "src")
        n = src.numel()
        if slots is not None:
            self._check_device_tensor(slots, torch.int32, "slots", n)
        _lib.check(_lib.lib().agarcl_batch_save_states(self._h, _vp(pool.data_ptr()), n_slots, _vp(src.data_ptr() if n else None),
                                                       _vp(slots.data_ptr()) if slots is not None and n else None, n, _vp(stream)))

    def restore_states(self, pool, slot_of, stream=0):
        """instance i <- pool slot slot_of[i] wherever slot_of[i] >= 0 (int32 CUDA tensor of N entries); enqueued on `stream`,
        no host wait.  Returns a view of the library-owned result u8 [N] (0 not requested, 1 restored, 2 rejected: the slot
        index is out of range or the slot was not saved from this configuration), which the next restore overwrites."""
        n_slots = self._check_pool(pool)
        self._check_device_tensor(slot_of, torch.int32, "slot_of", self.N)
        r = _vp()
        _lib.check(_lib.lib().agarcl_batch_restore_states(self._h, _vp(pool.data_ptr()), n_slots, _vp(slot_of.data_ptr()),
                                                          C.byref(r), _vp(stream)))
        return self._tensor(r.value, (self.N,), "|u1")

    def set_start_states(self, pool, start_slot=None, stream=0):
        """start-state table: from now on every reset of instance i (reset, reset_device and the auto-reset of step_autoreset)
        with start_slot[i] >= 0 begins the new episode in the game of pool slot start_slot[i], on the instance's own draw stream,
        instead of spawning a fresh one (include/agarcl_b200.h, agarcl_batch_set_start_states).  start_slot: int32 CUDA tensor
        of N entries (-1: spawn), copied on `stream`.  The batch holds on to the pool while it is set; slots saved into it later
        are read as they are when a reset runs.  pool None: every reset spawns again."""
        if pool is None:
            _lib.check(_lib.lib().agarcl_batch_set_start_states(self._h, None, 0, None, _vp(stream)))
            self._start_pool = None
            return
        n_slots = self._check_pool(pool)
        self._check_device_tensor(start_slot, torch.int32, "start_slot", self.N)
        _lib.check(_lib.lib().agarcl_batch_set_start_states(self._h, _vp(pool.data_ptr()), n_slots, _vp(start_slot.data_ptr()),
                                                            _vp(stream)))
        self._start_pool = pool

    def start_result(self):
        """view of the library-owned result u8 [N] of the latest reset with a start-state table: 0 not reset or spawned (slot
        -1), 1 started from its slot, 2 slot rejected (out of range, not saved from this configuration, or a mode outside the
        set) and spawned instead"""
        r = _vp()
        _lib.check(_lib.lib().agarcl_batch_start_result(self._h, C.byref(r)))
        return self._tensor(r.value, (self.N,), "|u1")

    # ---- Go-Explore cell archive (include/agarcl_b200.h, agarcl_batch_set_archive)
    def set_archive(self, pool, cells_per_side=None, agent=0, select=True, seed=0):
        """attaches a cleared archive whose entry e is pool slot e: every step_autoreset then files each game under its cell
        (agent `agent`'s position on a cells_per_side^2 grid x log2 of its mass), keeps the best game of every cell in the pool
        and, with select, starts every reset in a cell drawn with weight 1 / (1 + isqrt(times chosen)).  Needs set_autoreset
        first; synchronises the device.  The batch holds on to the pool while attached.  pool None detaches the archive."""
        if pool is None:
            _lib.check(_lib.lib().agarcl_batch_set_archive(self._h, None, 0, None))
            if getattr(self, "_archive_select", False):
                self._start_pool = None
            self._archive_pool, self._archive_select = None, False
            return
        n_slots = self._check_pool(pool)
        if cells_per_side is None:
            raise _lib.AgarclError("cells_per_side is needed to attach an archive")
        cfg = ArchiveCfg(cells_per_side=int(cells_per_side), agent=int(agent), select=int(bool(select)), pad=0,
                         seed=int(seed) & 0xFFFFFFFFFFFFFFFF)
        _lib.check(_lib.lib().agarcl_batch_set_archive(self._h, _vp(pool.data_ptr()), n_slots, C.byref(cfg)))
        if select or getattr(self, "_archive_select", False):  # (an archive that selected gave the table back)
            self._start_pool = pool if select else None
        self._archive_pool = pool
        self._archive_select = bool(select)

    def archive(self):
        """zero-copy device views of the archive: per instance cell_of (i32, -1 none), base_score (f64), base_length (i64); per
        key [32 n^2] key_entry (i32, -1 none) and visits (u32); per entry [K] entry_key, entry_score, entry_length, entry_chosen
        (u32); counters (u64 [3]: used, dropped, improved)"""
        a = Archive()
        _lib.check(_lib.lib().agarcl_batch_archive(self._h, C.byref(a)))
        N, n_keys, K = self.N, int(a.keys), int(a.entries)
        spec = {"cell_of": (N, "<i4"), "base_score": (N, "<f8"), "base_length": (N, "<i8"), "key_entry": (n_keys, "<i4"),
                "visits": (n_keys, "<u4"), "entry_key": (K, "<i4"), "entry_score": (K, "<f8"), "entry_length": (K, "<i8"),
                "entry_chosen": (K, "<u4"), "counters": (3, "<u8")}
        return {k: self._tensor(getattr(a, k), (n,), t) for k, (n, t) in spec.items()}

    # ---- pictures of game states (include/agarcl_b200.h, agarcl_batch_draw)
    def draw(self, src=None, size=256, view="arena", out=None, stream=0):
        """RGB pictures uint8 [n, size, size, 3] of the current states, drawn on the device (enqueued on `stream`, no host
        wait).  view "arena": the whole arena of instance src[k]; "agent": the observation window of image src[k] = instance * A
        + agent.  src: int32 CUDA tensor, or None for every instance (N pictures) or every agent (N * A).  A source out of range
        gives an all-zero picture.  out: a preallocated contiguous uint8 CUDA tensor [n, size, size, 3] to draw into."""
        if view not in DRAW_VIEWS:
            raise _lib.AgarclError(f"unknown view {view!r}: 'arena' or 'agent'")
        if src is None:
            n = self.N * (self.A if view == "agent" else 1)
        else:
            self._check_device_tensor(src, torch.int32, "src")
            n = src.numel()
        size = int(size)
        if out is None:
            out = torch.empty((n, size, size, 3), dtype=torch.uint8, device=self._device)
        else:
            self._check_device_tensor(out, torch.uint8, "out")
            if tuple(out.shape) != (n, size, size, 3):
                raise _lib.AgarclError(f"out must be [{n}, {size}, {size}, 3], got {list(out.shape)}")
        if n == 0:  # (an empty tensor has no device address to check)
            return out
        _lib.check(_lib.lib().agarcl_batch_draw(self._h, DRAW_VIEWS[view], size, _vp(src.data_ptr()) if src is not None else None,
                                                n, _vp(out.data_ptr()), _vp(stream)))
        return out

    # ---- the pixel observation (include/agarcl_b200.h, cfg.pixel_obs)
    def _pixels(self, final):
        p, f, shape = _vp(), _vp(), (C.c_int64 * 4)()
        _lib.check(_lib.lib().agarcl_batch_pixels(self._h, C.byref(p), C.byref(f), C.byref(shape)))
        ptr = f.value if final else p.value
        if not ptr:
            raise _lib.AgarclError("no final pictures: set_autoreset(keep_final_obs=True) with cfg.pixel_obs")
        return self._tensor(ptr, tuple(shape), "|u1")

    def pixels(self):
        """zero-copy device view uint8 [N*A, S, S, 3] of every agent's picture (cfg.pixel_obs = S), rewritten by every step, reset
        and restore: the picture agarcl_batch_draw's agent view draws, with the players the step respawned still dead"""
        return self._pixels(False)

    def final_pixels(self):
        """zero-copy device view uint8 [N*A, S, S, 3] of the pictures the reset instances of the last step_autoreset ended their
        episode on (set_autoreset(keep_final_obs=True))"""
        return self._pixels(True)

    # ---- built-in bot policies for agents (include/agarcl_b200.h, agarcl_batch_bot_actions)
    def bot_actions(self, types, out=None, target=None):
        """what a built-in bot would do for every agent on the current state, computed on the device on torch's current stream
        (no host wait, the state is not touched).  Returns (dxdy f32 [N*A, 2], act i32 [N*A], status u8 [N*A]) device tensors
        that go straight into set_actions_device / step.  types: a bot type (BOT_HUNGRY .. BOT_AGGRESSIVE_SHY) for every agent,
        or an int32 CUDA tensor [N*A] with -1 for an agent to skip: its dxdy and act are not written.  dxdy = (target - location) / 10,
        not clamped.  status: 0 skipped, 1 decided, 2 no pellet to go for (dxdy 0), 3 the agent is dead (dxdy 0), 4 not a bot
        type.  out: preallocated (dxdy, act, status) tensors to write into (new ones start at zero).  target: an f32 CUDA tensor
        [N*A, 2] that also receives the targets in world coordinates."""
        NA, dev = self.N * self.A, self._device
        if isinstance(types, torch.Tensor):
            self._check_device_tensor(types, torch.int32, "types", NA)
        else:
            cache = self.__dict__.setdefault("_bot_types", {})
            if int(types) not in cache:
                cache[int(types)] = torch.full((NA,), int(types), dtype=torch.int32, device=dev)
            types = cache[int(types)]
        if out is None:
            out = (torch.zeros((NA, 2), dtype=torch.float32, device=dev), torch.zeros(NA, dtype=torch.int32, device=dev),
                   torch.zeros(NA, dtype=torch.uint8, device=dev))
        dxdy, act, status = out
        self._check_device_tensor(dxdy, torch.float32, "dxdy", 2 * NA)
        self._check_device_tensor(act, torch.int32, "act", NA)
        self._check_device_tensor(status, torch.uint8, "status", NA)
        if target is not None:
            self._check_device_tensor(target, torch.float32, "target", 2 * NA)
        _lib.check(_lib.lib().agarcl_batch_bot_actions(
            self._h, _vp(types.data_ptr()), _vp(dxdy.data_ptr()), _vp(act.data_ptr()),
            _vp(target.data_ptr()) if target is not None else None, _vp(status.data_ptr()),
            _vp(torch.cuda.current_stream(dev).cuda_stream)))
        return dxdy, act, status

    # ---- mixed-task batches (include/agarcl_b200.h, cfg.task_modes)
    def set_tasks(self, mode, max_steps=None, stream=0):
        """the task each instance's NEXT reset plays: mode (int32 CUDA tensor of N entries, -1 keeps the pending mode) and
        max_steps (int32 CUDA tensor of N entries or None: every pending limit kept; -1 the set_autoreset limit, 0 none).
        Checked on the device, enqueued on `stream`, no host wait.  Returns a view of the library-owned result u8 [N] (0 nothing
        set, 1 set, 2 rejected: mode not in task_modes or limit < -1), which the next call overwrites."""
        self._check_device_tensor(mode, torch.int32, "mode", self.N)
        if max_steps is not None:
            self._check_device_tensor(max_steps, torch.int32, "max_steps", self.N)
        r = _vp()
        _lib.check(_lib.lib().agarcl_batch_set_tasks(self._h, _vp(mode.data_ptr()), _vp(max_steps.data_ptr()) if max_steps is not None else None,
                                                     C.byref(r), _vp(stream)))
        return self._tensor(r.value, (self.N,), "|u1")

    def tasks(self):
        """zero-copy int32 device views [N] of the task state: mode and max_steps of the current episode, next_mode and
        next_max_steps of the next"""
        t = _TasksStruct()
        _lib.check(_lib.lib().agarcl_batch_tasks(self._h, C.byref(t)))
        return {k: self._tensor(getattr(t, k), (self.N,), "<i4") for k in ("mode", "max_steps", "next_mode", "next_max_steps")}

    def set_task_sizes(self, bots=None, pellets=None, viruses=None, stream=0):
        """the game sizes each instance's NEXT reset plays: bots (mode 0), pellets and viruses, each an int32 CUDA tensor of N
        entries or None (every pending value kept); an entry of -1 keeps that value.  cfg.num_bots / num_pellets / num_viruses
        are the maxima.  Checked on the device, enqueued on `stream`, no host wait.  Returns a view of the library-owned result
        u8 [N] (0 nothing set, 1 set, 2 rejected: a value outside [0, maximum] or a bot count the batch's player order does not
        allow; a rejected instance keeps all its pending sizes), which the next call overwrites."""
        ptrs = []
        for name, t in (("bots", bots), ("pellets", pellets), ("viruses", viruses)):
            if t is not None:
                self._check_device_tensor(t, torch.int32, name, self.N)
            ptrs.append(_vp(t.data_ptr()) if t is not None else None)
        r = _vp()
        _lib.check(_lib.lib().agarcl_batch_set_task_sizes(self._h, *ptrs, C.byref(r), _vp(stream)))
        return self._tensor(r.value, (self.N,), "|u1")

    def task_sizes(self):
        """zero-copy int32 device views [N] of the game sizes: bots, pellets and viruses of the current episode, next_bots,
        next_pellets and next_viruses of the next"""
        t = _TaskSizesStruct()
        _lib.check(_lib.lib().agarcl_batch_task_sizes(self._h, C.byref(t)))
        return {k: self._tensor(getattr(t, k), (self.N,), "<i4") for k, _ in _TaskSizesStruct._fields_}

    # ---- parity / snapshot transport
    def download_state(self, i):
        sv = StateView(self.layout)
        _lib.check(_lib.lib().agarcl_batch_download_state(self._h, i, sv.ptr))
        return sv

    def upload_state(self, i, sv):
        if sv.blob.size != self.layout.stride:
            raise _lib.AgarclError(f"the state must be {self.layout.stride} bytes (one instance of this batch), got {sv.blob.size}")
        _lib.check(_lib.lib().agarcl_batch_upload_state(self._h, i, sv.ptr))

    def save_env_state(self, i, path):
        _lib.check(_lib.lib().agarcl_batch_save_env_state(self._h, i, str(path).encode()))

    def load_env_state(self, i, path, lossless=False):
        _lib.check(_lib.lib().agarcl_batch_load_env_state(self._h, i, str(path).encode(), int(lossless)))

    def set_replay(self, i, draws):
        d = np.ascontiguousarray(draws, dtype=np.float32)
        _lib.check(_lib.lib().agarcl_batch_set_replay(self._h, i, d.ctypes.data_as(_vp), d.size))

    # ---- zero-copy device views
    def obs_view(self):
        return _CudaView(self._obs_ptr, self.obs_shape, "<i2" if self.obs_dtype == np.int16 else "<i4", self)

    def rewards_view(self):
        return _CudaView(self._rew_ptr, (self.N * self.A,), "<f8", self)

    def dones_view(self):
        return _CudaView(self._done_ptr, (self.N * self.A,), "|u1", self)

    def obs_tensor(self):
        return self._tensor(self._obs_ptr, self.obs_shape, np.dtype(self.obs_dtype).str)

    def rewards_tensor(self):
        return self._tensor(self._rew_ptr, (self.N * self.A,), "<f8")

    def dones_tensor(self):
        return self._tensor(self._done_ptr, (self.N * self.A,), "|u1")
