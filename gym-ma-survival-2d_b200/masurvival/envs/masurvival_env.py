"""Batched, B200-resident drop-in for the reference's pseudo-gym environment.

Mirrors the API of `masurvival.envs.masurvival_env.MaSurvival`
(reference masurvival/envs/masurvival_env.py:241-895): same config dict and
merge rule (env:49-54), same observation keys and per-env shapes
(env:391-447), same action encoding `MultiDiscrete([3,3,3,2,2,2])` per agent
(env:449-453), same `reset()` / `step()` / `flush_stats()` names -- every
array just gains a leading batch dimension N.  All arithmetic happens in
libmasurv.so (hand-written sm_100a CUDA) behind a ctypes C ABI; tensors come
back as zero-copy torch views (DLPack) of library-owned HBM and stay valid
until the next step().  There is no CPU path.
"""
import numpy as np

from .. import _lib
from ..config import merge_config, pack_config
from . import spaces


class MaSurvivalVec:
    """N independent masurvival environments advanced by one kernel launch.

    Parameters
    ----------
    config : dict or None   reference-style nested config (env:140-238)
    num_envs : int          batch size N
    device : int            CUDA device ordinal
    seed : int              Philox key (the reference's unseeded numpy RNG,
                            env:50, is replaced by counter-based Philox4x32-10)
    env_offset : int        global index of env 0 (multi-GPU sharding)
    auto_reset : bool|str   True: reset finished envs inside step(); the returned
                            observation is then the first one of the new
                            episode (rewards/dones still describe the old).
                            'terminal': same, and step()'s info dict carries
                            info['terminal_observation'] (rows valid where done),
                            lidar_frac / lidar_hit included when lidars are
                            configured (one more lidar scan per step, in this
                            mode only)
    max_episode_steps : int|None  step limit (vector-env extension; None or 0:
                            none).  An episode that has run this many steps
                            without ending on the last one is truncated:
                            step()'s info['truncated'] flags it, episode_return /
                            episode_length rows are valid where done | truncated,
                            and auto_reset treats it like a finished episode
                            (auto_reset=False only flags it: see reset_envs)
    """

    metadata = {'render_modes': ['rgb_array'], 'render_fps': 30}

    def __init__(self, config=None, num_envs=1, device=0, seed=0, env_offset=0, auto_reset=True, max_episode_steps=None):
        self.config, self._continuous_melee = merge_config(config)
        self._rec = pack_config(self.config, self._continuous_melee, auto_reset=auto_reset,
                                max_episode_steps=max_episode_steps or 0)
        self.num_envs = int(num_envs)
        self.device = int(device)
        self.auto_reset = bool(auto_reset)
        self._terminal = int(self._rec['auto_reset']) == 2
        self._h = _lib.Handle(self._rec, self.num_envs, device, seed, env_offset)
        self.observation_space = self.compute_obs_space()
        self.action_space = self.compute_action_space()
        self.steps = 0
        self._act_buf = None
        self._done_bool = None
        self._trunc_bool = None
        self._host_obs = None
        self._mask_buf = None

    # ---- reference properties (env:245-291) --------------------------------
    @property
    def n_agents(self):
        return int(self._rec['n_agents'])

    @property
    def n_heals(self):
        return int(self._rec['n_heals'])

    @property
    def n_boxes(self):
        return int(self._rec['n_boxes'])

    @property
    def box_ownership(self):
        return bool(self._rec['box_ownership'])

    @property
    def has_teams(self):
        return bool(self._rec['teams'])

    def entity_keys(self):
        ks = {'others'}
        if self.n_heals > 0:
            ks |= {'heals', 'heal_slot'}
        if self.n_boxes > 0:
            ks |= {'boxes', 'box_items', 'box_slot'}
        return ks

    # ---- spaces (env:391-453) ----------------------------------------------
    def obs_shapes(self):
        A, B, H = self.n_agents, self.n_boxes, self.n_heals
        S = 8 + (1 if self.has_teams else 0)
        d = {'agent': (A, S), 'zone': (A, 6), 'others': (A, A - 1, S), 'others_mask': (A, A - 1)}
        if H > 0:
            d.update({'heals': (A, H, 2), 'heals_mask': (A, H), 'heal_slot': (A, 1, 1), 'heal_slot_mask': (A, 1)})
        if B > 0:
            d.update({'boxes': (A, B, 11), 'boxes_mask': (A, B), 'box_items': (A, B, 10),
                      'box_items_mask': (A, B), 'box_slot': (A, 1, 8), 'box_slot_mask': (A, 1)})
        L = int(self._rec['lidar_n'])
        if L > 0:
            d.update({'lidar_frac': (A, L), 'lidar_hit': (A, L)})
        return d

    def compute_obs_space(self):
        return spaces.Dict({k: spaces.Box(float('-inf'), float('inf'), shape=s)
                            for k, s in self.obs_shapes().items() if k != 'lidar_hit'})

    def compute_action_space(self):
        return spaces.Tuple((spaces.MultiDiscrete([3, 3, 3, 2, 2, 2]),) * self.n_agents)

    # ---- tensors -----------------------------------------------------------
    def _obs(self, prefix=''):
        """Observation dict with the reference's per-env shapes and a leading
        N.  `zone`, `heals`, `boxes`, `box_items` are identical for every
        observer (env:550,559,582,610 tile them): they are stored once per env
        and returned as stride-0 expanded views."""
        h, A = self._h, self.n_agents
        x = {}
        for k in self.obs_shapes():
            t = h.tensor(prefix + k)
            if k in ('zone', 'heals', 'boxes', 'box_items'):
                t = t.unsqueeze(1).expand(t.shape[0], A, *t.shape[1:])
            x[k] = t
        return x

    def _stream(self):
        import torch
        return torch.cuda.current_stream(self.device).cuda_stream

    def reset(self, seed=None, return_info=False, options=None):
        """BaseEnv.reset (env:59-74) for all N envs (the `seed` argument is
        ignored, as in the reference).  options={'reset_mask': m} resets only
        the envs `m` selects (see reset_envs)."""
        if options and 'reset_mask' in options:
            obs = self.reset_envs(options['reset_mask'])
            return (obs, {}) if return_info else obs
        self._h.reset(self._stream())
        self.steps = 0
        obs = self._obs()
        return (obs, {}) if return_info else obs

    def reset_envs(self, mask):
        """BaseEnv.reset (env:59-74) for the chosen envs only; the others are left untouched.  `mask`: a
        CUDA bool or uint8 tensor of N elements on this device (used in place, no host synchronisation: a
        step and a reset_envs can be captured together in a CUDA graph), a host boolean array of N, or a
        sequence of env indices.  A reset env starts its next episode (the draws an auto-reset would make);
        its rewards, dones and truncated flags are zeroed; its episode_return / episode_length rows, which
        describe the last finished episode, are kept, and flush_stats() does not count the interrupted
        episode.  Returns the observation dict."""
        import torch
        N, dev = self.num_envs, f'cuda:{self.device}'
        if isinstance(mask, torch.Tensor) and mask.is_cuda:
            if mask.device.index != self.device:
                raise ValueError(f'reset mask lives on {mask.device}, the environments on {dev}')
            if mask.dtype not in (torch.bool, torch.uint8) or mask.numel() != N:
                raise ValueError(f'a device reset mask must be a bool or uint8 tensor of {N} elements')
            m = mask.reshape(N).contiguous()
        else:
            arr = np.asarray(mask.cpu() if isinstance(mask, torch.Tensor) else mask)
            if arr.dtype == np.bool_:
                if arr.size != N:
                    raise ValueError(f'a host reset mask must have {N} elements')
                m = arr.reshape(N)
            elif arr.size == 0 or np.issubdtype(arr.dtype, np.integer):
                idx = arr.reshape(-1).astype(np.int64)
                if ((idx < 0) | (idx >= N)).any():
                    raise ValueError(f'env indices must be in 0..{N - 1}')
                m = np.zeros(N, dtype=np.bool_)
                m[idx] = True
            else:
                raise ValueError('reset mask: a bool/uint8 CUDA tensor, a host boolean array or a sequence of env indices')
            m = torch.from_numpy(np.ascontiguousarray(m)).to(dev)
        self._mask_buf = m     # keep alive until the stream has consumed it
        self._h.reset_envs(m.data_ptr(), self._stream())
        return self._obs()

    def step(self, actions):
        """BaseEnv.step (env:76-90).  `actions`: integer array-like
        [N, A, 6]; a CUDA uint8 torch tensor is consumed in place, anything
        else is validated and copied to the device."""
        import torch
        N, A = self.num_envs, self.n_agents
        if isinstance(actions, torch.Tensor) and actions.is_cuda and actions.dtype == torch.uint8:
            # consumed in place; out-of-range components are clamped by the kernel (the
            # reference asserts, env:80: validating on the device would cost a sync per step)
            if actions.device.index != self.device:
                raise ValueError(f'actions live on {actions.device}, the environments on cuda:{self.device}')
            a = actions.contiguous()
        else:
            arr = np.asarray(actions.cpu() if isinstance(actions, torch.Tensor) else actions)
            arr = arr.reshape(N, A, 6)
            nvec = np.array([3, 3, 3, 2, 2, 2])
            assert ((arr >= 0) & (arr < nvec)).all(), f'Invalid action {actions}.'  # env:80
            a = torch.as_tensor(arr.astype(np.uint8)).to(f'cuda:{self.device}', non_blocking=False)
        if a.numel() != N * A * 6:
            raise ValueError(f'actions must have {N}x{A}x6 elements')
        self._act_buf = a  # keep alive until the stream has consumed it
        self._h.step(a.data_ptr(), self._stream())
        self.steps += 1
        info = {'terminal_observation': self._obs('terminal_')} if self._terminal else {}
        # per-env episode statistics (rows valid where done, or done | truncated under a step limit): what a
        # trainer logs at episode end
        info['episode_return'] = self._h.tensor('episode_return')
        info['episode_length'] = self._h.tensor('episode_length')
        if self._rec['max_episode_steps'] > 0:
            trunc = self._h.tensor('truncated')
            if self._trunc_bool is None or self._trunc_bool.data_ptr() != trunc.data_ptr():
                self._trunc_bool = trunc.view(torch.bool)
            info['truncated'] = self._trunc_bool
        for k in ('immune', 'br_over', 'br_results'):
            if self._h.has_tensor(k):
                info[k] = self._h.tensor(k)
        dones = self._h.tensor('dones')
        if self._done_bool is None or self._done_bool.data_ptr() != dones.data_ptr():
            self._done_bool = dones.view(torch.bool)      # zero-copy: uint8 0/1 reinterpreted, no per-step allocation
        return self._obs(), self._h.tensor('rewards'), self._done_bool, info

    def step_host(self, actions, rewards_out=None, dones_out=None):
        """End-to-end step from HOST buffers: actions uint8[N,A,6] (numpy or
        pinned torch CPU tensor) -> rewards float32[N,A], dones uint8[N] in
        host memory; copies happen inside the call."""
        a, rewards_out, dones_out = self._host_args(actions, rewards_out, dones_out)
        self._h.step_host(self._ptr(a), self._ptr(rewards_out), self._ptr(dones_out), self._stream())
        self.steps += 1
        return rewards_out, dones_out

    @staticmethod
    def _ptr(t):
        return t.ctypes.data if isinstance(t, np.ndarray) else t.data_ptr()

    @staticmethod
    def _check_host(name, t, dtype, numel):
        """raw pointers cross the C ABI: dtype, size and contiguity are checked here"""
        import torch
        if isinstance(t, np.ndarray):
            ok = t.dtype == np.dtype(dtype) and t.size == numel and t.flags['C_CONTIGUOUS']
        elif isinstance(t, torch.Tensor):
            ok = (not t.is_cuda) and t.dtype == getattr(torch, np.dtype(dtype).name) and t.numel() == numel and t.is_contiguous()
        else:
            ok = False
        if not ok:
            raise ValueError(f'{name} must be a C-contiguous host {np.dtype(dtype).name} array/tensor with {numel} elements')

    def _host_args(self, actions, rewards_out, dones_out):
        N, A = self.num_envs, self.n_agents
        a = np.ascontiguousarray(actions, dtype=np.uint8) if isinstance(actions, np.ndarray) else actions
        if rewards_out is None:
            rewards_out = np.empty((N, A), dtype=np.float32)
        if dones_out is None:
            dones_out = np.empty((N,), dtype=np.uint8)
        self._check_host('actions', a, np.uint8, N * A * 6)
        self._check_host('rewards_out', rewards_out, np.float32, N * A)
        self._check_host('dones_out', dones_out, np.uint8, N)
        return a, rewards_out, dones_out

    def host_obs_buffer(self, pinned=True):
        """A host buffer for step_host_obs (page-locked by default) and the dict of
        zero-copy numpy views into it, one per observation key (library layout:
        `zone/heals/boxes/box_items` once per env, see _obs)."""
        import torch
        nbytes = self._h.obs_host_bytes()
        buf = torch.empty(nbytes, dtype=torch.uint8)
        if pinned:
            buf = buf.pin_memory()
        raw = buf.numpy()
        views, N, A = {}, self.num_envs, self.n_agents
        for k, shp in self.obs_shapes().items():
            off = self._h.obs_host_offset(k)
            if k in ('zone', 'heals', 'boxes', 'box_items'):
                shp = shp[1:]
            dt = np.int32 if k == 'lidar_hit' else np.float32
            n = int(np.prod(shp)) * N
            views[k] = raw[off:off + 4 * n].view(dt).reshape((N,) + tuple(shp))
        return buf, views

    def step_host_obs(self, actions, obs_buf, rewards_out=None, dones_out=None):
        """step_host that also lands the observations in `obs_buf` (from
        host_obs_buffer()): H2D actions, kernels, D2H rewards/dones/observations."""
        a, rewards_out, dones_out = self._host_args(actions, rewards_out, dones_out)
        self._check_host('obs_buf', obs_buf, np.uint8, self._h.obs_host_bytes())
        self._h.step_host_obs(self._ptr(a), self._ptr(rewards_out), self._ptr(dones_out), self._ptr(obs_buf), self._stream())
        self.steps += 1
        return rewards_out, dones_out

    def step_host_async(self, actions, rewards_out, dones_out, obs_buf=None):
        """Enqueue a host-buffer step and return; step_host_wait() blocks until the host
        buffers are complete.  Lets a caller keep several env groups in flight."""
        a, rewards_out, dones_out = self._host_args(actions, rewards_out, dones_out)
        if obs_buf is not None:
            self._check_host('obs_buf', obs_buf, np.uint8, self._h.obs_host_bytes())
        self._h.step_host_async(self._ptr(a), self._ptr(rewards_out), self._ptr(dones_out),
                                None if obs_buf is None else self._ptr(obs_buf), self._stream())
        self.steps += 1

    def step_host_wait(self):
        self._h.step_host_wait()

    def observe(self):
        self._h.observe(self._stream())
        return self._obs()

    def tile_plan(self):
        """How this batch is tiled onto the GPU (msv_tile_plan): envs per thread block of the step
        kernel, its blocks and threads per block, and whether the observation kernel consumes the step
        kernel's tiles as they finish.  No counterpart in the reference (it steps one env at a time)."""
        return self._h.tile_plan()

    # ---- stats (env:471-508) -------------------------------------------------
    def flush_stats(self):
        """Sum of the reference's per-env flush_stats() dict over all envs."""
        s = self._h.flush_stats()
        n = 2 if self.has_teams else self.n_agents
        out = {f'reward{i}': float(s['reward'][i]) for i in range(n)}
        out.update({f'kills{i}': int(s['kills'][i]) for i in range(n)})
        out['steps'] = int(s['steps'])
        out['heals_used'] = int(s['heals_used'])
        out['boxes_placed'] = int(s['boxes_placed'])
        out['episodes'] = int(s['episodes'])
        return out

    # ---- parity injection / checkpoint --------------------------------------
    def get_state(self, first=0, count=None):
        return self._h.get_state(first, count)

    def set_state(self, states, first=0):
        self._h.set_state(states, first)

    def bytes_per_env_step(self):
        return self._h.bytes_per_env_step()

    def obs_bytes_per_env(self):
        return self._h.obs_bytes_per_env()

    def kernel_launches(self):
        return self._h.kernel_launches()

    def device_bytes(self):
        return self._h.device_bytes()

    def render(self, mode='rgb_array', first=0, count=None, height=256, width=256, lidar=False, out=None):
        """Top-down RGB pictures of environments [first, first+count) as drawn by the library's
        render kernel from the device state: a CUDA uint8 tensor [count, height, width, 3] (row 0 at
        the top, +y up), enqueued on the current torch stream after the last step.  Under auto_reset,
        a finished environment shows the first state of its new episode.  `lidar=True` draws the rays
        (lidars must be configured).  Pass `out` (same shape, contiguous, on this device) to reuse a
        buffer.  Colours: masurvival._lib.render_palette(), named by _lib.RENDER_COLOURS."""
        import torch
        if mode != 'rgb_array':
            raise NotImplementedError(f'render mode {mode!r}: only rgb_array is supported (there is no window)')
        count = self.num_envs - first if count is None else count
        if count < 1 or height < 1 or width < 1:
            raise ValueError(f'render: count, height and width must be positive (got {count}, {height}, {width})')
        shape = (int(count), int(height), int(width), 3)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=f'cuda:{self.device}')
        elif not (isinstance(out, torch.Tensor) and out.is_cuda and out.device.index == self.device
                  and out.dtype == torch.uint8 and tuple(out.shape) == shape and out.is_contiguous()):
            raise ValueError(f'out must be a contiguous uint8 tensor of shape {shape} on cuda:{self.device}')
        self._h.render(first, count, out, _lib.MSV_RENDER_LIDAR if lidar else 0, self._stream())
        return out

    def close(self):
        self._h.close()


class MaSurvival(MaSurvivalVec):
    """Single-environment view with the reference's exact call shapes:
    `reset()` -> dict of numpy float32 arrays, `step(actions)` ->
    `(obs, float32[A], bool, {})` with `actions` a tuple of A 6-tuples."""

    def __init__(self, config=None, device=0, seed=0):
        super().__init__(config, num_envs=1, device=device, seed=seed, auto_reset=False)

    def _np_obs(self, obs):
        return {k: v[0].cpu().numpy() for k, v in obs.items()}

    def reset(self, seed=None, return_info=False, options=None):
        obs = self._np_obs(super().reset())
        return (obs, {}) if return_info else obs

    def render(self, mode='rgb_array', height=256, width=256, lidar=False):
        """numpy uint8[height, width, 3] picture of the environment (gym's rgb_array convention)."""
        return super().render(mode, 0, 1, height, width, lidar)[0].cpu().numpy()

    def step(self, actions):
        actions = tuple(a for a in actions)
        assert self.action_space.contains(actions), f'Invalid action {actions}.'
        obs, rew, done, info = super().step(np.asarray(actions, dtype=np.int64).reshape(1, self.n_agents, 6))
        return self._np_obs(obs), rew[0].cpu().numpy(), bool(done[0].item()), {}   # env:90 returns an empty info dict
