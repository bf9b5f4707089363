"""msv_render / MaSurvivalVec.render on the device: every pixel equal to the numpy reference
(tests/render_reference.py) on rolled-out and crafted states, the render leaves the simulation untouched
(state, observations and the k_step -> k_obs2 hand-off), bad arguments are refused without a launch, the
single-environment API, and demo.py's frame dumper."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import obs_cases as oc
import parity
import render_reference as rr
from parity import random_actions

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [(1, 1), (5, 7), (7, 5), (64, 64), (256, 256), (200, 300)]      # (height, width)
# (name, variant, overrides); configs with lidars are drawn with the lidar flag off and on
CONFIGS = [
    ('2v2', '2v2', {}),
    ('ffa', 'ffa', {}),
    ('1v1_heal_only', '1v1_heal_only', {}),
    ('teams_owned', '2v2', {'boxes': {'ownership': True}}),
    ('ffa_lidar', 'ffa_lidar', {}),
]


def _user(variant, over):
    return parity.apply_overrides(parity.variant(variant), oc._merge(oc.FAST, over))


def _check_frames(env, seen, tag):
    """render every size and range of env's current state; compare with the reference of get_state()"""
    import torch
    torch.cuda.synchronize()
    N = env.num_envs
    states = env.get_state()
    rec = env._rec
    lidar_flags = (False, True) if int(rec['lidar_n']) > 0 else (False,)
    frac = env._h.tensor('lidar_frac').cpu().numpy() if int(rec['lidar_n']) > 0 else None
    ranges = [(0, N), (N // 3, N // 3), (N - 1, 1)]
    for lidar in lidar_flags:
        for H, W in SIZES:
            want = {}
            for first, count in ranges:
                got = env.render(first=first, count=count, height=H, width=W, lidar=lidar).cpu().numpy()
                assert got.shape == (count, H, W, 3)
                for q in range(count):
                    e = first + q
                    if e not in want:
                        idx = rr.render_indices(rec, states[e], H, W, frac[e] if lidar else None)
                        seen.update(np.unique(idx).tolist())
                        want[e] = rr.palette()[idx]
                    if not np.array_equal(got[q], want[e]):
                        bad = np.argwhere((got[q] != want[e]).any(-1))
                        j, i = bad[0]
                        raise AssertionError(f'{tag} lidar={lidar} {H}x{W} env {e}: {len(bad)} pixels differ, first '
                                             f'({j}, {i}) device {got[q][j, i]} reference {want[e][j, i]}')


def test_render_matches_reference():
    import torch
    from masurvival import _lib
    from masurvival.envs import MaSurvivalVec
    seen = set()
    N = 37                                              # a multiple of no tile or block size
    for name, variant, over in CONFIGS:
        env = MaSurvivalVec(_user(variant, over), N, seed=11, auto_reset=True)
        rng = np.random.default_rng(5)
        env.reset()
        torch.cuda.synchronize()
        base = env.get_state(0, 1)[0]
        for t in range(90):                             # zone phases advance, agents die, items lie on the floor
            env.step(random_actions(rng, N, env.n_agents))
            if t in (30, 89):
                _check_frames(env, seen, f'{name} step {t + 1}')
        cases = oc.observation_states(env._rec, base, rng)
        env.set_state(np.array([cases[e % len(cases)][1] for e in range(N)]))
        env.observe()                                   # the lidar scan of the injected states
        _check_frames(env, seen, f'{name} crafted')
        assert env._h.overflow_events() == 0
        env.close()
    missing = [_lib.RENDER_COLOURS[k] for k in range(len(_lib.RENDER_COLOURS)) if k not in seen]
    assert not missing, missing


def test_render_is_read_only_and_keeps_the_hand_off():
    import torch
    from masurvival.envs import MaSurvivalVec
    N = 1000
    envs = [MaSurvivalVec(parity.variant('2v2'), N, seed=3, auto_reset=True) for _ in range(2)]
    plan = envs[0].tile_plan()
    assert plan['blocks'] > 1 and plan['observation_hand_off'], plan
    g = torch.Generator(device='cuda:0')
    g.manual_seed(9)
    for env in envs:
        env.reset()
    buf = torch.empty((N, 64, 64, 3), dtype=torch.uint8, device='cuda:0')
    for t in range(200):
        a = torch.randint(0, 2, (N, 4, 6), dtype=torch.uint8, device='cuda:0', generator=g)
        a[..., :3] = torch.randint(0, 3, (N, 4, 3), dtype=torch.uint8, device='cuda:0', generator=g)
        outs = [env.step(a) for env in envs]
        envs[0].render(count=N, height=64, width=64, out=buf)
        assert torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[1][2]), t
    torch.cuda.synchronize()
    for k in outs[0][0]:                                        # the last step's observations
        assert torch.equal(outs[0][0][k], outs[1][0][k]), k
    for k in outs[0][3]:
        assert torch.equal(outs[0][3][k], outs[1][3][k]), k
    assert envs[0].kernel_launches() - envs[1].kernel_launches() == 200
    s0, s1 = envs[0].get_state(), envs[1].get_state()
    assert s0.tobytes() == s1.tobytes()
    assert envs[0]._h.overflow_events() == 0 and envs[1]._h.overflow_events() == 0
    for env in envs:
        env.close()


def test_render_counts_one_launch():
    from masurvival.envs import MaSurvivalVec
    env = MaSurvivalVec(parity.variant('2v2'), 20, seed=1)
    env.reset()
    n = env.kernel_launches()
    env.render(count=20, height=16, width=16)
    assert env.kernel_launches() == n + 1
    env.close()


def test_bad_arguments_are_refused():
    import torch
    from masurvival import _lib
    from masurvival.envs import MaSurvivalVec
    N = 10
    env, twin = (MaSurvivalVec(parity.variant('2v2'), N, seed=4, auto_reset=True) for _ in range(2))
    env.reset(); twin.reset()
    L, h = _lib.load(), env._h.h
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device='cuda:0')    # larger than any of the requests below
    p = ctypes.c_void_p(buf.data_ptr())
    n0 = env.kernel_launches()
    bad = [(None, 0, 1, 8, 8, 0, p), (h, 0, 1, 8, 8, 0, None), (h, -1, 1, 8, 8, 0, p), (h, 0, 0, 8, 8, 0, p),
           (h, 5, 6, 8, 8, 0, p), (h, 0, N + 1, 8, 8, 0, p), (h, 0, 1, 0, 8, 0, p), (h, 0, 1, 4097, 1, 0, p),
           (h, 0, 1, 8, 0, 0, p), (h, 0, 1, 1, 4097, 0, p), (h, 0, 1, 8, 8, 2, p),
           (h, 0, 1, 8, 8, _lib.MSV_RENDER_LIDAR, p)]          # no lidars in 2v2
    for args in bad:
        assert L.msv_render(*args, None) == -1, args             # MSV_ERR_INVALID
    assert env.kernel_launches() == n0                          # nothing was launched
    with pytest.raises(_lib.MasurvError):
        env.render(first=-1, count=1)
    with pytest.raises(_lib.MasurvError):
        env.render(first=5, count=6)
    with pytest.raises(_lib.MasurvError):
        env.render(count=1, height=4097, width=1)
    with pytest.raises(_lib.MasurvError):
        env.render(count=1, lidar=True)
    with pytest.raises(ValueError):
        env.render(count=0)
    for wrong in (torch.zeros((1, 8, 8, 3), dtype=torch.float32, device='cuda:0'),
                  torch.zeros((1, 8, 8, 3), dtype=torch.uint8),
                  torch.zeros((2, 8, 8, 3), dtype=torch.uint8, device='cuda:0'),
                  torch.zeros((1, 8, 16, 3), dtype=torch.uint8, device='cuda:0')[:, :, ::2],
                  torch.zeros((1, 8, 8, 4), dtype=torch.uint8, device='cuda:0')):
        with pytest.raises(ValueError):
            env.render(count=1, height=8, width=8, out=wrong)
    assert env.kernel_launches() == n0
    with pytest.raises(NotImplementedError):
        env.render('human')
    rng = np.random.default_rng(2)
    for _ in range(30):                                         # the handle keeps stepping as its twin does
        a = random_actions(rng, N, 4)
        r0, r1 = env.step(a)[1], twin.step(a)[1]
        assert torch.equal(r0, r1)
    assert env.get_state().tobytes() == twin.get_state().tobytes()
    env.close(); twin.close()


def test_single_env_render():
    from masurvival.envs import MaSurvival, MaSurvivalVec
    env = MaSurvival(parity.variant('2v2'), seed=7)
    env.reset()
    rng = np.random.default_rng(1)
    for _ in range(10):
        env.step(tuple(tuple(int(v) for v in a) for a in random_actions(rng, 1, 4)[0]))
    img = env.render('rgb_array')
    assert isinstance(img, np.ndarray) and img.shape == (256, 256, 3) and img.dtype == np.uint8
    assert np.array_equal(img, MaSurvivalVec.render(env, count=1)[0].cpu().numpy())
    assert np.array_equal(img, rr.render_reference(env._rec, env.get_state()[0], 256, 256))
    assert 'rgb_array' in MaSurvival.metadata['render_modes']
    with pytest.raises(NotImplementedError):
        env.render('human')
    env.close()


def _demo(tmp_path, extra):
    cfg = tmp_path / 'cfg.json'
    cfg.write_text(json.dumps(parity.variant('2v2')))      # a user config names its melee class (env:309-312)
    cmd = [sys.executable, os.path.join(ROOT, 'gym-ma-survival-2d_b200', 'demo.py'), '-c', str(cfg), '-n', '8',
           '--max-steps', '20', '--benchmark'] + extra
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


def test_demo_dumps_frames(tmp_path):
    out = tmp_path / 'frames'
    text = _demo(tmp_path, ['--dump-frames', str(out), '--frame-envs', '4'])
    assert re.search(r'Performance test results: [0-9.eE+-]+, [0-9.eE+-]+', text), text
    for key in ('reward0', 'kills0', 'steps', 'heals_used', 'boxes_placed', 'episodes'):
        assert f"'{key}'" in text, (key, text)
    files = sorted(os.listdir(out))
    assert files == [f'frame_{t:05d}.png' for t in range(1, 21)], files
    for f in files:
        assert rr.read_png(str(out / f)).shape == (512, 512, 3)
    out3 = tmp_path / 'every3'
    _demo(tmp_path, ['--dump-frames', str(out3), '--frame-envs', '3', '--frame-size', '32', '--frame-every', '3'])
    files = sorted(os.listdir(out3))
    assert files == [f'frame_{t:05d}.png' for t in range(3, 21, 3)], files
    assert rr.read_png(str(out3 / files[0])).shape == (64, 64, 3)      # 3 envs: 2 per row, 2 rows
