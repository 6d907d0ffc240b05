"""ctypes binding of libagarcl_b200.so (include/agarcl_b200.h).  Fails loudly when the library is
missing or a call fails: there is no CPU path in this package."""
import ctypes as C
import os

from ._abi import Archive, ArchiveCfg, Cfg, Layout

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libagarcl_b200.so")

_vp = C.c_void_p
_lib = None

# argtypes of every function include/agarcl_b200.h declares; all return int except the two in _RESTYPES
_PROTOTYPES = {
    "agarcl_make_layout": [C.POINTER(Cfg), C.POINTER(Layout)],
    "agarcl_batch_create": [C.POINTER(Cfg), C.POINTER(_vp)],
    "agarcl_batch_destroy": [_vp],
    "agarcl_batch_get_layout": [_vp, C.POINTER(Layout)],
    "agarcl_batch_seed": [_vp, _vp],
    "agarcl_batch_reset": [_vp, _vp, _vp],
    "agarcl_batch_set_actions": [_vp, _vp, _vp, C.c_int, _vp],
    "agarcl_batch_step": [_vp, _vp],
    "agarcl_batch_obs": [_vp, C.POINTER(_vp), C.POINTER(C.c_int64 * 4), C.POINTER(C.c_int32)],
    "agarcl_batch_rewards": [_vp, C.POINTER(_vp)],
    "agarcl_batch_dones": [_vp, C.POINTER(_vp)],
    "agarcl_batch_step_host": [_vp, _vp, _vp, _vp, _vp, _vp],
    "agarcl_batch_reset_device": [_vp, _vp, _vp],
    "agarcl_batch_set_autoreset": [_vp, C.c_int32, C.c_int32, C.c_int32],
    "agarcl_batch_step_autoreset": [_vp, _vp],
    "agarcl_batch_episode": [_vp, _vp],
    "agarcl_snapshot_slot_bytes": [C.POINTER(Cfg), C.POINTER(C.c_int64)],
    "agarcl_batch_save_states": [_vp, _vp, C.c_int64, _vp, _vp, C.c_int32, _vp],
    "agarcl_batch_restore_states": [_vp, _vp, C.c_int64, _vp, C.POINTER(_vp), _vp],
    "agarcl_batch_set_start_states": [_vp, _vp, C.c_int64, _vp, _vp],
    "agarcl_batch_start_result": [_vp, C.POINTER(_vp)],
    "agarcl_batch_set_archive": [_vp, _vp, C.c_int64, C.POINTER(ArchiveCfg)],
    "agarcl_batch_archive": [_vp, C.POINTER(Archive)],
    "agarcl_batch_set_tasks": [_vp, _vp, _vp, C.POINTER(_vp), _vp],
    "agarcl_batch_tasks": [_vp, _vp],
    "agarcl_batch_set_task_sizes": [_vp, _vp, _vp, _vp, C.POINTER(_vp), _vp],
    "agarcl_batch_task_sizes": [_vp, _vp],
    "agarcl_batch_draw": [_vp, C.c_int32, C.c_int32, _vp, C.c_int32, _vp, _vp],
    "agarcl_batch_pixels": [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_int64 * 4)],
    "agarcl_batch_bot_actions": [_vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "agarcl_batch_mirror": [_vp, C.POINTER(_vp), C.POINTER(C.c_int64 * 4), C.POINTER(C.c_int32)],
    "agarcl_batch_sync_mirror": [_vp, _vp],
    "agarcl_batch_step_mirror": [_vp, _vp, _vp, _vp, _vp],
    "agarcl_batch_mirror_stats": [_vp, C.POINTER(C.c_uint64 * 4)],
    "agarcl_batch_mirror_timing": [_vp, C.POINTER(C.c_uint64 * 4)],
    "agarcl_batch_step_lists": [_vp, _vp, _vp, _vp, _vp, _vp],
    "agarcl_batch_lists_expand": [_vp, C.c_int32, _vp],
    "agarcl_batch_download_state": [_vp, C.c_int32, _vp],
    "agarcl_batch_upload_state": [_vp, C.c_int32, _vp],
    "agarcl_batch_save_env_state": [_vp, C.c_int32, C.c_char_p],
    "agarcl_batch_load_env_state": [_vp, C.c_int32, C.c_char_p, C.c_int],
    "agarcl_snapshot_write": [C.POINTER(Cfg), C.POINTER(Layout), _vp, C.c_char_p],
    "agarcl_snapshot_read": [C.POINTER(Cfg), C.POINTER(Layout), _vp, C.c_char_p, C.c_int],
    "agarcl_batch_set_replay": [_vp, C.c_int32, _vp, C.c_int32],
    "agarcl_batch_render": [_vp, _vp],
    "agarcl_batch_ram": [_vp, C.POINTER(_vp), C.POINTER(C.c_int64 * 3)],
    "agarcl_batch_render_ram": [_vp, _vp],
    "agarcl_batch_ram_host": [_vp, _vp],
    "agarcl_batch_launches_per_step": [_vp],
    "agarcl_batch_flags": [_vp, _vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32 * 32)],
    "agarcl_selftest_std_sort": [_vp, C.c_int32, _vp],
    "agarcl_batch_costs": [_vp, _vp, _vp],
    "agarcl_batch_set_timing": [_vp, C.c_int],
    "agarcl_batch_get_timing": [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32)],
    "agarcl_mt19937_draws": [C.c_uint64, _vp, C.c_int32],
    "agarcl_last_error": [],
    "agarcl_version": [],
}
_RESTYPES = {"agarcl_last_error": C.c_char_p, "agarcl_version": C.c_char_p}
SYMBOLS = list(_PROTOTYPES)


class AgarclError(RuntimeError):
    """C-ABI call failed (the reference raises EnvironmentException -> RuntimeError, bindings.cpp)."""


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is not built: run `python -m agarcl_b200.build` "
                              "(agarcl_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, argtypes in _PROTOTYPES.items():
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, C.c_int)
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
