"""ctypes loader for libmasurv.so (the C ABI declared in include/masurv.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device
is visible when an environment is created, this raises."""
import ctypes
import os

import numpy as np

from .config import CONFIG_DT, STATE_DT, STATS_DT

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('MSV_LIB') or os.path.join(_HERE, 'libmasurv.so')   # MSV_LIB: development override

MSV_OK = 0
ERRORS = {-1: 'MSV_ERR_INVALID', -2: 'MSV_ERR_CUDA', -3: 'MSV_ERR_NO_DEVICE',
          -4: 'MSV_ERR_NAME', -5: 'MSV_ERR_ALLOC'}

EXPORTS = [
    'msv_abi_version', 'msv_sizeof_config', 'msv_sizeof_env_state', 'msv_sizeof_stats',
    'msv_default_config', 'msv_create', 'msv_destroy', 'msv_reset', 'msv_reset_envs', 'msv_step',
    'msv_step_host', 'msv_step_host_obs', 'msv_step_host_async', 'msv_step_host_wait', 'msv_obs_host_bytes',
    'msv_obs_host_offset', 'msv_device_bytes', 'msv_tensor', 'msv_tensor_info', 'msv_get_state', 'msv_set_state',
    'msv_observe', 'msv_flush_stats', 'msv_bytes_per_env_step', 'msv_kernel_bytes_per_env', 'msv_obs_bytes_per_env', 'msv_kernel_launches', 'msv_tile_plan', 'msv_plan_tile',
    'msv_last_error', 'msv_philox4x32', 'msv_render', 'msv_render_palette',
]

MSV_RENDER_LIDAR = 1
# the entries of msv_render_palette(), in the library's order (include/masurv.h)
RENDER_COLOURS = ('background', 'floor', 'floor_outside_zone', 'zone_ring', 'next_zone_ring', 'wall', 'heal',
                  'box_item', 'box') + tuple(f'agent{i}' for i in range(8)) + ('team0', 'team1', 'heading', 'lidar_ray')


class MasurvError(RuntimeError):
    pass


def render_palette():
    """The colours msv_render draws with: uint8[n, 3], row k is RENDER_COLOURS[k] (no device needed)."""
    L = load()
    out = np.zeros((64, 3), dtype=np.uint8)
    n = L.msv_render_palette(out.ctypes.data, out.shape[0])
    if n < 0:
        check(n)
    return out[:n].copy()


_lib = None


def load():
    """dlopen libmasurv.so and declare the signatures.  Works without a GPU
    (only msv_create needs one)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MasurvError(
            f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(nvcc, sm_100a). There is no CPU fallback.')
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, u64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64
    L.msv_abi_version.restype = ctypes.c_int
    for f in ('msv_sizeof_config', 'msv_sizeof_env_state', 'msv_sizeof_stats'):
        getattr(L, f).restype = i64
    L.msv_default_config.argtypes = [vp]
    L.msv_create.argtypes = [vp, i32, i32, u64, i64, ctypes.POINTER(vp)]
    L.msv_destroy.argtypes = [vp]
    L.msv_reset.argtypes = [vp, vp]
    L.msv_reset_envs.argtypes = [vp, vp, vp]
    L.msv_step.argtypes = [vp, vp, vp]
    L.msv_step_host.argtypes = [vp, vp, vp, vp, vp]
    L.msv_step_host_obs.argtypes = [vp, vp, vp, vp, vp, vp]
    L.msv_step_host_async.argtypes = [vp, vp, vp, vp, vp, vp]
    L.msv_step_host_wait.argtypes = [vp]
    L.msv_obs_host_bytes.argtypes = [vp]
    L.msv_obs_host_bytes.restype = i64
    L.msv_obs_host_offset.argtypes = [vp, ctypes.c_char_p]
    L.msv_obs_host_offset.restype = i64
    L.msv_device_bytes.argtypes = [vp]
    L.msv_device_bytes.restype = i64
    L.msv_debug_kernel_timing.argtypes = [vp, ctypes.c_int, vp, vp]
    L.msv_tensor.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(vp)]
    L.msv_tensor_info.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(vp), ctypes.POINTER(i32),
                                  ctypes.POINTER(i64), ctypes.POINTER(i64), ctypes.POINTER(i32)]
    L.msv_get_state.argtypes = [vp, i32, i32, vp]
    L.msv_set_state.argtypes = [vp, i32, i32, vp]
    L.msv_observe.argtypes = [vp, vp]
    L.msv_flush_stats.argtypes = [vp, vp]
    L.msv_bytes_per_env_step.argtypes = [vp]
    L.msv_bytes_per_env_step.restype = i64
    L.msv_kernel_bytes_per_env.argtypes = [vp, i32]
    L.msv_kernel_bytes_per_env.restype = i64
    L.msv_obs_bytes_per_env.argtypes = [vp]
    L.msv_obs_bytes_per_env.restype = i64
    L.msv_kernel_launches.argtypes = [vp]
    L.msv_kernel_launches.restype = i64
    L.msv_tile_plan.argtypes = [vp, vp]
    L.msv_plan_tile.argtypes = [vp, i32, i32, i64, vp]
    L.msv_last_error.argtypes = [vp]
    L.msv_last_error.restype = ctypes.c_char_p
    L.msv_philox4x32.argtypes = [vp, vp, vp]
    L.msv_render.argtypes = [vp, i32, i32, i32, i32, ctypes.c_uint32, vp, vp]
    L.msv_render_palette.argtypes = [vp, i32]
    L.msv_debug_step_kernel.argtypes = [vp, vp, vp]
    L.msv_debug_obs_kernel.argtypes = [vp, vp]
    L.msv_debug_overflow.argtypes = [vp]
    L.msv_debug_overflow.restype = i64
    L.msv_debug_check_failures.argtypes = [vp, ctypes.POINTER(i64)]
    L.msv_debug_check_failures.restype = i64
    if L.msv_abi_version() != 2:
        raise MasurvError('libmasurv.so ABI version mismatch')
    for name, dt in (('msv_sizeof_config', CONFIG_DT), ('msv_sizeof_env_state', STATE_DT),
                     ('msv_sizeof_stats', STATS_DT)):
        if getattr(L, name)() != dt.itemsize:
            raise MasurvError(f'{name}: library says {getattr(L, name)()}, header parser says {dt.itemsize}')
    _lib = L
    return L


def check(rc, handle=None):
    if rc != MSV_OK:
        msg = load().msv_last_error(handle)
        raise MasurvError(f'{ERRORS.get(rc, rc)}: {msg.decode() if msg else ""}')


_PyCapsule_New = ctypes.pythonapi.PyCapsule_New
_PyCapsule_New.restype = ctypes.py_object
_PyCapsule_New.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p]


class Handle:
    """Owns one msv_handle (one batch of environments on one GPU)."""

    def __init__(self, cfg_rec, num_envs, device=0, seed=0, env_offset=0):
        L = load()
        self.cfg = np.array(cfg_rec, dtype=CONFIG_DT).reshape(1)
        self.num_envs = int(num_envs)
        self.device = int(device)
        h = ctypes.c_void_p()
        check(L.msv_create(self.cfg.ctypes.data, self.num_envs, self.device, int(seed), int(env_offset),
                           ctypes.byref(h)))
        self.h = h
        self._tensors = {}

    def close(self):
        """msv_destroy.  Tensors already handed out stay valid: the library keeps the
        device memory they alias until the last of them is garbage-collected."""
        if getattr(self, 'h', None):
            self._tensors.clear()
            load().msv_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def tensor(self, name):
        """Zero-copy torch view of a library-owned device tensor (DLPack)."""
        if name not in self._tensors:
            import torch
            m = ctypes.c_void_p()
            check(load().msv_tensor(self.h, name.encode(), ctypes.byref(m)), self.h)
            cap = _PyCapsule_New(m, b'dltensor', None)
            self._tensors[name] = torch.from_dlpack(cap)
        return self._tensors[name]

    def has_tensor(self, name):
        p = ctypes.c_void_p()
        return load().msv_tensor_info(self.h, name.encode(), ctypes.byref(p), None, None, None, None) == 0

    def reset(self, stream=0):
        check(load().msv_reset(self.h, stream), self.h)

    def reset_envs(self, mask_ptr, stream=0):
        """msv_reset_envs: `mask_ptr` is a device pointer to uint8[num_envs] (the caller checks it)."""
        check(load().msv_reset_envs(self.h, mask_ptr, stream), self.h)

    def observe(self, stream=0):
        check(load().msv_observe(self.h, stream), self.h)

    def step(self, actions_dev_ptr, stream=0):
        check(load().msv_step(self.h, actions_dev_ptr, stream), self.h)

    def step_kernel_only(self, actions_dev_ptr, stream=0):
        check(load().msv_debug_step_kernel(self.h, actions_dev_ptr, stream), self.h)

    def observe_only(self, stream=0):
        check(load().msv_debug_obs_kernel(self.h, stream), self.h)

    def render(self, first, count, out, flags=0, stream=0):
        """msv_render into `out`, a contiguous CUDA uint8 tensor [count, H, W, 3] (the caller checks it)."""
        check(load().msv_render(self.h, int(first), int(count), int(out.shape[1]), int(out.shape[2]), int(flags),
                                out.data_ptr(), stream), self.h)

    def step_host(self, actions, rewards, dones, stream=0):
        check(load().msv_step_host(self.h, actions, rewards, dones, stream), self.h)

    def step_host_obs(self, actions, rewards, dones, obs, stream=0):
        check(load().msv_step_host_obs(self.h, actions, rewards, dones, obs, stream), self.h)

    def step_host_async(self, actions, rewards, dones, obs=None, stream=0):
        check(load().msv_step_host_async(self.h, actions, rewards, dones, obs, stream), self.h)

    def step_host_wait(self):
        check(load().msv_step_host_wait(self.h), self.h)

    def obs_host_bytes(self):
        return int(load().msv_obs_host_bytes(self.h))

    def obs_host_offset(self, name):
        return int(load().msv_obs_host_offset(self.h, name.encode()))

    def device_bytes(self):
        return int(load().msv_device_bytes(self.h))

    def kernel_timing(self, enable):
        """debug: start (True) / stop (False) CUDA-event timing of the kernels of step(); stopping
        returns (mean ms of [k_step, k_obs2, k_lidar], number of steps recorded)."""
        out = (ctypes.c_double * 3)()
        n = ctypes.c_int64()
        check(load().msv_debug_kernel_timing(self.h, 1 if enable else 0, out, ctypes.byref(n)), self.h)
        return [float(x) for x in out], int(n.value)

    def get_state(self, first=0, count=None):
        count = self.num_envs - first if count is None else count
        out = np.zeros(count, dtype=STATE_DT)
        check(load().msv_get_state(self.h, first, count, out.ctypes.data), self.h)
        return out

    def set_state(self, states, first=0):
        buf = np.ascontiguousarray(np.asarray(states, dtype=STATE_DT).reshape(-1))
        check(load().msv_set_state(self.h, first, len(buf), buf.ctypes.data), self.h)

    def flush_stats(self):
        out = np.zeros(1, dtype=STATS_DT)
        check(load().msv_flush_stats(self.h, out.ctypes.data), self.h)
        return out[0]

    def overflow_events(self):
        return int(load().msv_debug_overflow(self.h))

    def check_failures(self):
        """(violations, source line of the last one) counted by a bounds-checked build (make CHECK=1);
        violations == -2 when the loaded library is not a checked build"""
        line = ctypes.c_int64()
        n = int(load().msv_debug_check_failures(self.h, ctypes.byref(line)))
        return n, int(line.value)

    def bytes_per_env_step(self):
        return int(load().msv_bytes_per_env_step(self.h))

    def kernel_bytes_per_env(self, which):
        """algorithmic HBM bytes per env-step of kernel `which` (0 k_step, 1 k_obs2, 2 k_lidar)"""
        return int(load().msv_kernel_bytes_per_env(self.h, which))

    def obs_bytes_per_env(self):
        return int(load().msv_obs_bytes_per_env(self.h))

    def kernel_launches(self):
        return int(load().msv_kernel_launches(self.h))

    def tile_plan(self):
        """how the batch is tiled onto the GPU (msv_tile_plan)"""
        out = (ctypes.c_int32 * 4)()
        check(load().msv_tile_plan(self.h, out), self.h)
        return {'envs_per_block': int(out[0]), 'blocks': int(out[1]), 'threads_per_block': int(out[2]),
                'observation_hand_off': bool(out[3])}
