"""MaSurvivalVec(..., obs_layout='flat'): the flat observation is a pure relayout of the dict one.  A flat
handle and a dict handle with the same config, seed and actions run in lock-step; every step the flat rows
must equal the concatenation of the dict handle's tensors, and every named key, step output and terminal
observation must be the same bits.  Also: the tile hand-off, CUDA graphs, host read-back, render and the
byte accounting in the flat layout."""
import numpy as np
import pytest

import obs_cases as oc
import parity

pytestmark = pytest.mark.gpu


def _user(name, over):
    return parity.apply_overrides(parity.variant(name), {k: dict(v) for k, v in over.items()})


# every entry of the config matrix (three capacity classes, 1-7 agents, partial observability, H = 0, B = 0,
# lidar), plus 2v2, ffa_lidar and 1v1_heal_only; N = 70 leaves the last tile ragged.  (id, user config, step
# limit): every case must end episodes within its 150 steps; 1v1_heal_only has no melee damage and its episodes
# outlast them, so its case ends them at a step limit
CASES = [(cid, _user('1v1', oc._merge(oc.FAST, over)), None) for cid, _, over, _ in oc.MATRIX] + [
    ('2v2', _user('2v2', {'safe_zone': {'cooldown': 8}, 'health': {'health': 30}}), None),
    ('ffa_lidar', _user('ffa_lidar', {'safe_zone': {'cooldown': 6}, 'health': {'health': 20}}), None),
    ('heal_only', _user('1v1_heal_only', {'safe_zone': {'cooldown': 8}}), 30),
]


def _pair(user, N, seed=3, **kw):
    from masurvival.envs import MaSurvivalVec
    return (MaSurvivalVec(user, N, seed=seed, obs_layout='dict', **kw),
            MaSurvivalVec(user, N, seed=seed, obs_layout='flat', **kw))


def _keys(env):
    return [k for k in env.obs_shapes() if k != 'lidar_hit']


def _concat(obs, keys, N, A):
    import torch
    return torch.cat([obs[k].reshape(N, A, -1) for k in keys], 2)


def _bits(t):
    import torch
    return t.contiguous().view(torch.int32)


def _same(a, b):
    import torch
    return torch.equal(_bits(a), _bits(b)) if a.dtype == torch.float32 else torch.equal(a, b)


def _check_obs(tag, ed, ef, od, of):
    """flat rows = concatenation of the dict tensors; every key through the flat handle's views = the dict key"""
    import torch
    N, A = ed.num_envs, ed.n_agents
    keys = _keys(ed)
    flat = ef.flat_obs()
    assert flat.shape == (N, A, sum(int(np.prod(s[1:])) for k, s in ed.obs_shapes().items() if k != 'lidar_hit'))
    assert torch.equal(_bits(flat), _bits(_concat(od, keys, N, A))), tag
    assert set(od) == set(of), tag
    for k in od:
        assert od[k].shape == of[k].shape and _same(od[k], of[k]), (tag, k)


def _check_outputs(tag, ed, ef, rd, rf, dd, df, infd, inff):
    import torch
    assert _same(rd, rf) and torch.equal(dd, df), tag
    for k in ('episode_return', 'episode_length', 'truncated'):
        if k in infd:
            assert _same(infd[k], inff[k]), (tag, k)


def _actions(g, N, A):
    import torch
    a = torch.empty((N, A, 6), dtype=torch.uint8, device='cuda')
    a[..., :3] = torch.randint(0, 3, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
    a[..., 3:] = torch.randint(0, 2, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
    return a


def _lockstep(user, mode, N=70, steps=150, T=None, seed=3):
    import torch
    ed, ef = _pair(user, N, seed=seed, auto_reset=mode, max_episode_steps=T)
    A, keys = ed.n_agents, _keys(ed)
    L = int(ed._rec['lidar_n'])
    D = ef.flat_obs().shape[2]
    _check_obs('reset', ed, ef, ed.reset(), ef.reset())
    g = torch.Generator(device='cuda'); g.manual_seed(seed)
    finished_total, prev_term = 0, None
    for t in range(steps):
        a = _actions(g, N, A)
        od, rd, dd, infd = ed.step(a)
        of, rf, df, inff = ef.step(a)
        tag = (mode, T, t)
        _check_obs(tag, ed, ef, od, of)
        _check_outputs(tag, ed, ef, rd, rf, dd, df, infd, inff)
        fin = dd | infd['truncated'] if 'truncated' in infd else dd.clone()
        finished_total += int(fin.sum())
        if mode == 'terminal':
            td, tf = infd['terminal_observation'], inff['terminal_observation']
            for k in td:
                assert _same(td[k], tf[k]), (tag, 'terminal', k)
            term = inff['terminal_observation_flat']
            assert torch.equal(_bits(term), _bits(_concat(td, keys, N, A))), tag
            if prev_term is not None:      # rows of envs that did not finish keep their bits (lidar columns aside)
                keep = ~fin
                assert torch.equal(_bits(term[keep][..., :D - L]), _bits(prev_term[keep][..., :D - L])), tag
            prev_term = term.clone()
        if t % 5 == 2:                     # reset_envs: a random mask (and the finished envs without auto-reset)
            m = torch.rand(N, device='cuda', generator=g) < 0.25
            if not mode:
                m |= fin
            _check_obs((tag, 'reset_envs'), ed, ef, ed.reset_envs(m), ef.reset_envs(m))
        elif not mode and fin.any():
            _check_obs((tag, 'reset_envs done'), ed, ef, ed.reset_envs(fin), ef.reset_envs(fin))
    # observe after set_state: the environments' states permuted
    states = ed.get_state()
    assert states.tobytes() == ef.get_state().tobytes()
    perm = np.random.default_rng(seed).permutation(N)
    ed.set_state(states[perm]); ef.set_state(states[perm])
    _check_obs('observe', ed, ef, ed.observe(), ef.observe())
    assert ed._h.overflow_events() == 0 and ef._h.overflow_events() == 0
    ed.close(); ef.close()
    return finished_total


@pytest.mark.parametrize('mode', [False, True, 'terminal'])
@pytest.mark.parametrize('cid,user,T', CASES, ids=[c[0] for c in CASES])
def test_flat_is_a_relayout(cid, user, T, mode):
    assert _lockstep(user, mode, T=T) > 0


@pytest.mark.parametrize('mode', [False, True, 'terminal'])
@pytest.mark.parametrize('name', ['2v2', 'ffa_lidar'])
def test_flat_is_a_relayout_with_step_limit(name, mode):
    user = [c[1] for c in CASES if c[0] == name][0]
    assert _lockstep(user, mode, N=45, steps=50, T=17) > 0


def test_flat_layout_shape_and_accounting():
    import torch
    for name, D in (('2v2', 160), ('1v1_heal_only', 37), ('ffa', 320), ('ffa_lidar', 352)):
        ed, ef = _pair(parity.variant(name), 36)
        ef.reset()
        A, L = ef.n_agents, int(ef._rec['lidar_n'])
        x = ef.flat_obs()
        assert x.shape == (36, A, D) and x.dtype == torch.float32 and x.is_contiguous() and x.data_ptr() % 16 == 0
        assert ef.flat_obs().data_ptr() == x.data_ptr()
        assert ef.obs_bytes_per_env() == A * (D - L) * 4
        assert ef._h.kernel_bytes_per_env(1) - ed._h.kernel_bytes_per_env(1) == ef.obs_bytes_per_env() - ed.obs_bytes_per_env()
        lay = ef.flat_obs_layout()
        assert list(lay) == _keys(ed)
        col = 0
        for k, (c0, shp) in lay.items():
            assert c0 == col, k
            assert torch.equal(_bits(x[:, :, c0:c0 + int(np.prod(shp))]), _bits(ef._obs()[k].reshape(36, A, -1))), k
            col += int(np.prod(shp))
        assert col == D
        assert ed.tile_plan() == ef.tile_plan()
        n0d, n0f = ed.kernel_launches(), ef.kernel_launches()
        a = torch.zeros((36, A, 6), dtype=torch.uint8, device='cuda')
        ed.step(a); ef.step(a)
        assert ed.kernel_launches() - n0d == ef.kernel_launches() - n0f
        ed.close(); ef.close()


@pytest.mark.parametrize('vname,steps', [('2v2', 60), ('ffa_lidar', 40)])
def test_flat_hand_off_multi_wave(vname, steps, monkeypatch):
    """a batch of several waves: the hand-off writes the same obs_flat as plain stream-ordered launches"""
    import torch
    from masurvival.envs import MaSurvivalVec
    from test_gpu_config_matrix import _multiwave_n
    over = {'safe_zone': {'cooldown': 10}, 'health': {'health': 20}}
    cfg = parity.apply_overrides(parity.variant(vname), over)
    rec = parity.make_config(vname, auto_reset=True, **over)
    N = _multiwave_n(rec, torch.cuda.get_device_properties(0).multi_processor_count)
    monkeypatch.delenv('MSV_NO_HANDOFF', raising=False)
    e1 = MaSurvivalVec(cfg, N, seed=11, obs_layout='flat')
    e0 = MaSurvivalVec(cfg, N, seed=11, obs_layout='dict')
    monkeypatch.setenv('MSV_NO_HANDOFF', '1')
    e2 = MaSurvivalVec(cfg, N, seed=11, obs_layout='flat')
    monkeypatch.delenv('MSV_NO_HANDOFF', raising=False)
    assert e1.tile_plan()['observation_hand_off'] and not e2.tile_plan()['observation_hand_off']
    assert e1.tile_plan() == e0.tile_plan()
    A = e1.n_agents
    g = torch.Generator(device='cuda'); g.manual_seed(2)
    e1.reset(); e2.reset(); e0.reset()
    dones = 0
    for t in range(steps):
        a = _actions(g, N, A)
        _, r1, d1, _ = e1.step(a)
        _, r2, d2, _ = e2.step(a)
        o0, _, _, _ = e0.step(a)
        assert torch.equal(_bits(e1.flat_obs()), _bits(e2.flat_obs())), t
        assert torch.equal(_bits(e1.flat_obs()), _bits(_concat(o0, _keys(e0), N, A))), t
        assert _same(r1, r2) and torch.equal(d1, d2)
        dones += int(d1.sum())
    assert dones > 0
    assert e1._h.overflow_events() == 0 and e2._h.overflow_events() == 0
    e1.close(); e2.close(); e0.close()


def test_flat_cuda_graph_step_and_reset_envs():
    """a CUDA graph of step + reset_envs in the flat layout replays to the eager run's obs_flat"""
    import torch
    from masurvival.envs import MaSurvivalVec
    N, T = 300, 30
    user = _user('ffa_lidar', {'safe_zone': {'cooldown': 6}, 'health': {'health': 15}})
    eg, ee = (MaSurvivalVec(user, N, seed=8, auto_reset=False, max_episode_steps=T, obs_layout='flat') for _ in range(2))
    A = eg.n_agents
    rng = np.random.default_rng(5)
    a_static = torch.zeros((N, A, 6), dtype=torch.uint8, device='cuda')

    def body(env):
        _, _, d, info = env.step(a_static)
        env.reset_envs(d | info['truncated'])

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eg.reset(); ee.reset()
        for _ in range(3):
            a_static.copy_(torch.as_tensor(parity.random_actions(rng, N, A)))
            body(eg); body(ee)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body(eg)
    for t in range(40):
        a_static.copy_(torch.as_tensor(parity.random_actions(rng, N, A)))
        graph.replay()
        body(ee)
        torch.cuda.synchronize()
        assert torch.equal(_bits(eg.flat_obs()), _bits(ee.flat_obs())), t
        assert torch.equal(eg._h.tensor('lidar_hit'), ee._h.tensor('lidar_hit')), t
    assert eg.get_state().tobytes() == ee.get_state().tobytes()
    eg.close(); ee.close()


@pytest.mark.parametrize('name', ['2v2', 'ffa_lidar'])
def test_flat_step_host_obs(name):
    """step_host_obs in the flat layout: the host views (as_strided from msv_tensor_info) equal the device views"""
    import torch
    from masurvival.envs import MaSurvivalVec
    N = 50
    env = MaSurvivalVec(_user(name, {'safe_zone': {'cooldown': 8}}), N, seed=4, obs_layout='flat')
    env.reset()
    A = env.n_agents
    buf, views = env.host_obs_buffer()
    assert set(views) == set(env.obs_shapes())
    rng = np.random.default_rng(1)
    for t in range(10):
        a = parity.random_actions(rng, N, A)
        env.step_host_obs(a, buf)
        torch.cuda.synchronize()
        for k, v in views.items():
            want = env._h.tensor(k).cpu().numpy()
            assert v.shape == want.shape and np.array_equal(v.view(np.int32), want.view(np.int32)), (t, k)
    env.close()


@pytest.mark.parametrize('name', ['ffa_lidar', 'a7_lidar'])
def test_flat_render_lidar(name):
    """k_render reads lidar_frac with the flat row stride: pictures identical to the dict layout's"""
    import torch
    user = [c[1] for c in CASES if c[0] == name][0]
    ed, ef = _pair(user, 12, seed=6, auto_reset=True)
    ed.reset(); ef.reset()
    A = ed.n_agents
    g = torch.Generator(device='cuda'); g.manual_seed(9)
    for t in range(6):
        a = _actions(g, 12, A)
        ed.step(a); ef.step(a)
        pd, pf = ed.render(lidar=True, height=96, width=96), ef.render(lidar=True, height=96, width=96)
        assert torch.equal(pd, pf), t
    ed.close(); ef.close()
