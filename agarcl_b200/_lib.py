"""ctypes binding of libagarcl_b200.so (include/agarcl_b200.h).  Fails loudly when the library is
missing or a call fails: there is no CPU path in this package."""
import ctypes as C
import os

from ._abi import Archive, ArchiveCfg, Cfg, Layout

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libagarcl_b200.so")

_vp = C.c_void_p
_lib = None

SYMBOLS = [
    "agarcl_make_layout", "agarcl_batch_create", "agarcl_batch_destroy", "agarcl_batch_get_layout",
    "agarcl_batch_seed", "agarcl_batch_reset", "agarcl_batch_set_actions", "agarcl_batch_step",
    "agarcl_batch_obs", "agarcl_batch_rewards", "agarcl_batch_dones", "agarcl_batch_step_host",
    "agarcl_batch_reset_device", "agarcl_batch_set_autoreset", "agarcl_batch_step_autoreset", "agarcl_batch_episode",
    "agarcl_snapshot_slot_bytes", "agarcl_batch_save_states", "agarcl_batch_restore_states",
    "agarcl_batch_set_start_states", "agarcl_batch_start_result", "agarcl_batch_set_archive", "agarcl_batch_archive",
    "agarcl_batch_set_tasks", "agarcl_batch_tasks", "agarcl_batch_draw", "agarcl_batch_bot_actions",
    "agarcl_batch_mirror", "agarcl_batch_sync_mirror", "agarcl_batch_step_mirror", "agarcl_batch_mirror_stats", "agarcl_batch_mirror_timing", "agarcl_batch_step_lists", "agarcl_batch_lists_expand",
    "agarcl_batch_download_state", "agarcl_batch_upload_state", "agarcl_batch_save_env_state", "agarcl_batch_load_env_state",
    "agarcl_snapshot_write", "agarcl_snapshot_read", "agarcl_batch_set_replay",
    "agarcl_batch_render", "agarcl_batch_ram", "agarcl_batch_ram_host", "agarcl_batch_render_ram", "agarcl_batch_launches_per_step", "agarcl_batch_flags", "agarcl_batch_costs", "agarcl_selftest_std_sort", "agarcl_batch_set_timing", "agarcl_batch_get_timing", "agarcl_mt19937_draws",
    "agarcl_last_error", "agarcl_version",
]


class AgarclError(RuntimeError):
    """C-ABI call failed (the reference raises EnvironmentException -> RuntimeError, bindings.cpp)."""


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is not built: run `python -m agarcl_b200.build` "
                              "(agarcl_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.agarcl_last_error.restype = C.c_char_p
        L.agarcl_version.restype = C.c_char_p
        L.agarcl_make_layout.argtypes = [C.POINTER(Cfg), C.POINTER(Layout)]
        L.agarcl_batch_create.argtypes = [C.POINTER(Cfg), C.POINTER(_vp)]
        L.agarcl_batch_destroy.argtypes = [_vp]
        L.agarcl_batch_get_layout.argtypes = [_vp, C.POINTER(Layout)]
        L.agarcl_batch_seed.argtypes = [_vp, _vp]
        L.agarcl_batch_reset.argtypes = [_vp, _vp, _vp]
        L.agarcl_batch_set_actions.argtypes = [_vp, _vp, _vp, C.c_int, _vp]
        L.agarcl_batch_step.argtypes = [_vp, _vp]
        L.agarcl_batch_obs.argtypes = [_vp, C.POINTER(_vp), C.POINTER(C.c_int64 * 4), C.POINTER(C.c_int32)]
        L.agarcl_batch_rewards.argtypes = [_vp, C.POINTER(_vp)]
        L.agarcl_batch_dones.argtypes = [_vp, C.POINTER(_vp)]
        L.agarcl_batch_step_host.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp]
        L.agarcl_batch_reset_device.argtypes = [_vp, _vp, _vp]
        L.agarcl_batch_set_autoreset.argtypes = [_vp, C.c_int32, C.c_int32, C.c_int32]
        L.agarcl_batch_step_autoreset.argtypes = [_vp, _vp]
        L.agarcl_batch_episode.argtypes = [_vp, _vp]
        L.agarcl_snapshot_slot_bytes.argtypes = [C.POINTER(Cfg), C.POINTER(C.c_int64)]
        L.agarcl_batch_save_states.argtypes = [_vp, _vp, C.c_int64, _vp, _vp, C.c_int32, _vp]
        L.agarcl_batch_restore_states.argtypes = [_vp, _vp, C.c_int64, _vp, C.POINTER(_vp), _vp]
        L.agarcl_batch_set_start_states.argtypes = [_vp, _vp, C.c_int64, _vp, _vp]
        L.agarcl_batch_start_result.argtypes = [_vp, C.POINTER(_vp)]
        L.agarcl_batch_set_archive.argtypes = [_vp, _vp, C.c_int64, C.POINTER(ArchiveCfg)]
        L.agarcl_batch_archive.argtypes = [_vp, C.POINTER(Archive)]
        L.agarcl_batch_set_tasks.argtypes = [_vp, _vp, _vp, C.POINTER(_vp), _vp]
        L.agarcl_batch_tasks.argtypes = [_vp, _vp]
        L.agarcl_batch_draw.argtypes = [_vp, C.c_int32, C.c_int32, _vp, C.c_int32, _vp, _vp]
        L.agarcl_batch_pixels.argtypes = [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_int64 * 4)]
        L.agarcl_batch_bot_actions.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.agarcl_batch_mirror.argtypes = [_vp, C.POINTER(_vp), C.POINTER(C.c_int64 * 4), C.POINTER(C.c_int32)]
        L.agarcl_batch_sync_mirror.argtypes = [_vp, _vp]
        L.agarcl_batch_step_mirror.argtypes = [_vp, _vp, _vp, _vp, _vp]
        L.agarcl_batch_mirror_stats.argtypes = [_vp, C.POINTER(C.c_uint64 * 4)]
        L.agarcl_batch_mirror_timing.argtypes = [_vp, C.POINTER(C.c_uint64 * 4)]
        L.agarcl_batch_step_lists.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp]
        L.agarcl_batch_lists_expand.argtypes = [_vp, C.c_int32, _vp]
        L.agarcl_batch_download_state.argtypes = [_vp, C.c_int32, _vp]
        L.agarcl_batch_upload_state.argtypes = [_vp, C.c_int32, _vp]
        L.agarcl_batch_save_env_state.argtypes = [_vp, C.c_int32, C.c_char_p]
        L.agarcl_batch_load_env_state.argtypes = [_vp, C.c_int32, C.c_char_p, C.c_int]
        L.agarcl_snapshot_write.argtypes = [C.POINTER(Cfg), C.POINTER(Layout), _vp, C.c_char_p]
        L.agarcl_snapshot_read.argtypes = [C.POINTER(Cfg), C.POINTER(Layout), _vp, C.c_char_p, C.c_int]
        L.agarcl_batch_set_replay.argtypes = [_vp, C.c_int32, _vp, C.c_int32]
        L.agarcl_batch_render.argtypes = [_vp, _vp]
        L.agarcl_batch_ram.argtypes = [_vp, C.POINTER(_vp), C.POINTER(C.c_int64 * 3)]
        L.agarcl_batch_render_ram.argtypes = [_vp, _vp]
        L.agarcl_batch_ram_host.argtypes = [_vp, _vp]
        L.agarcl_batch_launches_per_step.argtypes = [_vp]
        L.agarcl_batch_flags.argtypes = [_vp, _vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32 * 32)]
        L.agarcl_selftest_std_sort.argtypes = [_vp, C.c_int32, _vp]
        L.agarcl_batch_costs.argtypes = [_vp, _vp, _vp]
        L.agarcl_batch_set_timing.argtypes = [_vp, C.c_int]
        L.agarcl_batch_get_timing.argtypes = [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32)]
        L.agarcl_mt19937_draws.argtypes = [C.c_uint64, _vp, C.c_int32]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise AgarclError(lib().agarcl_last_error().decode() or f"agarcl error {rc}")


def make_layout(cfg):
    L = Layout()
    check(lib().agarcl_make_layout(C.byref(cfg), C.byref(L)))
    return L


def snapshot_slot_bytes(cfg):
    """bytes of one snapshot slot of configuration `cfg` (a multiple of 128; slot layout: include/agarcl_b200.h)"""
    n = C.c_int64()
    check(lib().agarcl_snapshot_slot_bytes(C.byref(cfg), C.byref(n)))
    return int(n.value)
