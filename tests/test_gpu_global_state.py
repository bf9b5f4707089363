"""MaSurvivalVec(..., global_state=True): the global-state row is what an omniscient observer sees, stored once.
Three handles run in lock-step with one seed and one action stream: P (partial observability, state on), O
(omniscient, state on) and O' (omniscient, state off).  Omniscience only changes which targets the cameras test,
so the step outputs agree bit for bit; P's row equals O's, and every key of it equals the matching piece of O''s
observation (the per-env keys from observer 0); the alive mask and the step count equal get_state()'s.  Also:
terminal capture, resets, injected states, the output off, the flat layout, CUDA graphs, two devices."""
import numpy as np
import pytest

import obs_cases as oc
import parity

pytestmark = pytest.mark.gpu


def _user(name, over):
    return parity.apply_overrides(parity.variant(name), {k: dict(v) for k, v in over.items()})


# every entry of the config matrix with partial observability forced on, plus 2v2, ffa_lidar and 1v1_heal_only
# (whose episodes outlast the run without melee damage: a step limit ends them); N = 70 leaves the last tile ragged
CASES = [(cid, _user('1v1', oc._merge(oc.FAST, over, oc.PARTIAL)), None) for cid, _, over, _ in oc.MATRIX] + [
    ('2v2', _user('2v2', {'safe_zone': {'cooldown': 8}, 'health': {'health': 30}, **oc.PARTIAL}), None),
    ('ffa_lidar', _user('ffa_lidar', {'safe_zone': {'cooldown': 6}, 'health': {'health': 20}, **oc.PARTIAL}), None),
    ('heal_only', _user('1v1_heal_only', {'safe_zone': {'cooldown': 8}, **oc.PARTIAL}), 30),
]


def _omni(user):
    return parity.apply_overrides({k: dict(v) for k, v in user.items()}, {'observation': {'omniscent': True}})


def _bits(t):
    import torch
    return t.contiguous().view(torch.int32)


def _same(a, b):
    import torch
    return torch.equal(_bits(a), _bits(b)) if a.dtype == torch.float32 else torch.equal(a, b)


def _actions(g, N, A):
    import torch
    a = torch.empty((N, A, 6), dtype=torch.uint8, device='cuda')
    a[..., :3] = torch.randint(0, 3, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
    a[..., 3:] = torch.randint(0, 2, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
    return a


def _pieces(env, obs):
    """the keys of the row that an omniscient observation holds: {key: [N, ...]} (per-env keys from observer 0)"""
    N, A = env.num_envs, env.n_agents
    out = {'agents': obs['agent'], 'zone': obs['zone'][:, 0]}
    if env.n_heals > 0:
        out.update({'heals': obs['heals'][:, 0], 'heals_mask': obs['heals_mask'][:, 0],
                    'heal_slot': obs['heal_slot'].reshape(N, A), 'heal_slot_mask': obs['heal_slot_mask'].reshape(N, A)})
    if env.n_boxes > 0:
        out.update({'boxes': obs['boxes'][:, 0], 'boxes_mask': obs['boxes_mask'][:, 0],
                    'box_items': obs['box_items'][:, 0], 'box_items_mask': obs['box_items_mask'][:, 0],
                    'box_slot': obs['box_slot'].reshape(N, A, 8), 'box_slot_mask': obs['box_slot_mask'].reshape(N, A)})
    return out


def _check_pieces(tag, env, obs, prefix='global_state', rows=None):
    """every key of env's row (the library's strided views) equals the observation's piece, in the selected rows"""
    for k, want in _pieces(env, obs).items():
        got = env._h.tensor(f'{prefix}_{k}')
        assert got.shape == want.shape, (tag, k, got.shape, want.shape)
        if rows is not None:
            got, want = got[rows], want[rows]
        assert _equal_bits(got, want), (tag, k)


def _equal_bits(a, b):
    import torch
    return torch.equal(_bits(a), _bits(b))


def _check_alive_steps(tag, env, states=None):
    import torch
    s = env.get_state() if states is None else states
    A = env.n_agents
    alive = torch.as_tensor(np.asarray(s['alive'])[:, :A].astype(np.float32))
    steps = torch.as_tensor(np.asarray(s['steps']).astype(np.float32)).reshape(-1, 1)
    assert torch.equal(env._h.tensor('global_state_agents_mask').cpu(), 1.0 - alive), tag
    assert torch.equal(env._h.tensor('global_state_steps').cpu(), steps), tag


def _layout_is_the_row(env):
    """state_layout() tiles the row in key order, and the library's views are the row's columns"""
    x = env.state()
    col = 0
    for k, (c0, shp) in env.state_layout().items():
        assert c0 == col, k
        w = int(np.prod(shp))
        assert _equal_bits(x[:, c0:c0 + w], env._h.tensor('global_state_' + k).reshape(env.num_envs, w)), k
        col += w
    assert col == x.shape[1] == env.state_space.shape[0]


def _triple(user, N, seed, **kw):
    from masurvival.envs import MaSurvivalVec
    return (MaSurvivalVec(user, N, seed=seed, global_state=True, **kw),
            MaSurvivalVec(_omni(user), N, seed=seed, global_state=True, **kw),
            MaSurvivalVec(_omni(user), N, seed=seed, **kw))


def _lockstep(user, mode, N=70, steps=120, T=None, seed=3):
    import torch
    P, O, Q = _triple(user, N, seed, auto_reset=mode, max_episode_steps=T)
    A = P.n_agents
    assert not P._rec['omniscient'] and O._rec['omniscient']
    envs = (P, O, Q)
    oq = Q.reset(); P.reset(); O.reset()
    _layout_is_the_row(P)
    _check_pieces('reset', P, oq)
    assert _equal_bits(P.state(), O.state())
    g = torch.Generator(device='cuda'); g.manual_seed(seed)
    finished_total = 0
    for t in range(steps):
        a = _actions(g, N, A)
        snap = P._h.tensor('terminal_global_state').clone() if mode == 'terminal' else None
        rp, ro, rq = (e.step(a) for e in envs)
        tag = (mode, T, t)
        for r in (ro, rp):
            assert _same(r[1], rq[1]) and torch.equal(r[2], rq[2]), tag
            for k in ('episode_return', 'episode_length', 'truncated'):
                if k in rq[3]:
                    assert _same(r[3][k], rq[3][k]), (tag, k)
        assert _equal_bits(P.state(), O.state()), tag
        _check_pieces(tag, P, rq[0])
        fin = rq[2] | rq[3]['truncated'] if 'truncated' in rq[3] else rq[2].clone()
        finished_total += int(fin.sum())
        if mode == 'terminal':
            term = rp[3]['terminal_state']
            assert _equal_bits(term, ro[3]['terminal_state']), tag
            _check_pieces((tag, 'terminal'), P, rq[3]['terminal_observation'], 'terminal_global_state', fin)
            assert _equal_bits(term[~fin], snap[~fin]), tag
        if t % 25 == 7:
            _check_alive_steps(tag, P)
        if t % 5 == 2 or (not mode and fin.any()):
            m = torch.rand(N, device='cuda', generator=g) < 0.25
            if not mode:
                m |= fin
            oq = Q.reset_envs(m); P.reset_envs(m); O.reset_envs(m)
            _check_pieces((tag, 'reset_envs'), P, oq)
            assert _equal_bits(P.state(), O.state()), tag
    for e in envs:
        assert e._h.overflow_events() == 0
        e.close()
    return finished_total


@pytest.mark.parametrize('mode', [False, True, 'terminal'])
@pytest.mark.parametrize('cid,user,T', CASES, ids=[c[0] for c in CASES])
def test_state_is_the_omniscient_observation(cid, user, T, mode):
    assert _lockstep(user, mode, T=T) > 0


@pytest.mark.parametrize('mode', [False, True, 'terminal'])
@pytest.mark.parametrize('name', ['2v2', 'ffa_lidar'])
def test_state_with_step_limit(name, mode):
    user = [c[1] for c in CASES if c[0] == name][0]
    assert _lockstep(user, mode, N=45, steps=50, T=17) > 0


@pytest.mark.parametrize('frac', [0.01, 0.5, 1.0])
def test_state_after_reset_envs(frac):
    import torch
    user = [c[1] for c in CASES if c[0] == '2v2'][0]
    P, O, Q = _triple(user, 300, 5, auto_reset=False)
    A = P.n_agents
    for e in (P, O, Q):
        e.reset()
    g = torch.Generator(device='cuda'); g.manual_seed(1)
    for t in range(30):
        a = _actions(g, 300, A)
        for e in (P, O, Q):
            e.step(a)
    m = torch.rand(300, device='cuda', generator=g) < frac
    if frac < 1.0:
        m[0] = True
    else:
        m[:] = True
    before = P.state().clone()
    oq = Q.reset_envs(m); P.reset_envs(m); O.reset_envs(m)
    _check_pieces(('reset_envs', frac), P, oq)
    assert _equal_bits(P.state(), O.state())
    assert _equal_bits(P.state()[~m], before[~m])
    _check_alive_steps('reset_envs', P)
    for e in (P, O, Q):
        e.close()


@pytest.mark.parametrize('cid,user,T', CASES, ids=[c[0] for c in CASES])
def test_state_of_injected_states(cid, user, T):
    """observe() after set_state of crafted states: dead first and last agents, a heal or box on top of an
    inventory, empty and full lists, the last zone phase"""
    import torch
    P, O, Q = _triple(user, 70, 9, auto_reset=False)
    P.reset(); O.reset(); Q.reset()
    base = P.get_state()
    rng = np.random.default_rng(4)
    states, tags = [], []
    for e in range(70):
        cases = oc.observation_states(P._rec, base[e], rng)
        tag, s = cases[e % len(cases)]
        states.append(s); tags.append(tag)
    assert len(set(tags)) == len(cases)
    states = np.array(states)
    for e in (P, O, Q):
        e.set_state(states)
    oq = Q.observe(); P.observe(); O.observe()
    _check_pieces(cid, P, oq)
    assert _equal_bits(P.state(), O.state())
    _check_alive_steps(cid, P, states)
    for e in (P, O, Q):
        e.close()


@pytest.mark.parametrize('name,mode,T', [('2v2', True, None), ('ffa_lidar', True, None), ('2v2', 'terminal', None),
                                         ('ffa', False, 20), ('1v1_heal_only', 'terminal', 25)])
def test_state_off_changes_nothing(name, mode, T):
    """a handle with the output and one without it: the same outputs, bit for bit; the launches differ by exactly
    the k_global_state launches; the tile plan (hand-off included) is the same"""
    import torch
    from masurvival.envs import MaSurvivalVec
    user = _user(name, {'safe_zone': {'cooldown': 8}, 'health': {'health': 25}})
    N = 1000
    on = MaSurvivalVec(user, N, seed=2, auto_reset=mode, max_episode_steps=T, global_state=True)
    off = MaSurvivalVec(user, N, seed=2, auto_reset=mode, max_episode_steps=T)
    assert on.tile_plan() == off.tile_plan()
    assert off._h.kernel_bytes_per_env(3) == 0
    assert on._h.kernel_bytes_per_env(3) > 4 * on.state().shape[1]
    assert on.bytes_per_env_step() - off.bytes_per_env_step() == on._h.kernel_bytes_per_env(3)
    assert not off._h.has_tensor('global_state') and not off._h.has_tensor('global_state_agents')
    per_step = 2 if mode == 'terminal' else 1
    extra = 1                                  # the enabling call writes the rows once
    oa, ob = on.reset(), off.reset()
    extra += 1
    for k in oa:
        assert _same(oa[k], ob[k]), k
    g = torch.Generator(device='cuda'); g.manual_seed(7)
    A = on.n_agents
    for t in range(60):
        a = _actions(g, N, A)
        ra, rb = on.step(a), off.step(a)
        extra += per_step
        for k in ra[0]:
            assert _same(ra[0][k], rb[0][k]), (t, k)
        assert _same(ra[1], rb[1]) and torch.equal(ra[2], rb[2]), t
        assert set(ra[3]) - set(rb[3]) <= {'terminal_state'}
        for k, v in rb[3].items():
            if isinstance(v, dict):
                for kk in v:
                    assert _same(ra[3][k][kk], v[kk]), (t, k, kk)
            else:
                assert _same(ra[3][k], v), (t, k)
        if t % 20 == 10:
            oa, ob = on.observe(), off.observe()
            extra += 1
    torch.cuda.synchronize()
    assert on.get_state().tobytes() == off.get_state().tobytes()
    assert on.kernel_launches() - off.kernel_launches() == extra
    assert on.tile_plan() == off.tile_plan()
    on.close(); off.close()


def test_state_hand_off_stays_on():
    """a batch of several waves with the tile hand-off: the state-on handle keeps the hand-off and writes the
    same observations as a state-off handle"""
    import torch
    from masurvival.envs import MaSurvivalVec
    from test_gpu_config_matrix import _multiwave_n
    over = {'safe_zone': {'cooldown': 10}, 'health': {'health': 20}}
    user = _user('2v2', over)
    rec = parity.make_config('2v2', auto_reset=True, **over)
    N = _multiwave_n(rec, torch.cuda.get_device_properties(0).multi_processor_count)
    on = MaSurvivalVec(user, N, seed=11, global_state=True)
    off = MaSurvivalVec(user, N, seed=11)
    assert on.tile_plan()['observation_hand_off'] and on.tile_plan() == off.tile_plan()
    on.reset(); off.reset()
    g = torch.Generator(device='cuda'); g.manual_seed(2)
    for t in range(40):
        a = _actions(g, N, on.n_agents)
        ra, rb = on.step(a), off.step(a)
        for k in ra[0]:
            assert _same(ra[0][k], rb[0][k]), (t, k)
        _check_pieces(t, on, rb[0])
    assert on._h.overflow_events() == 0
    on.close(); off.close()


def test_state_with_flat_layout():
    import torch
    from masurvival.envs import MaSurvivalVec
    user = _user('ffa_lidar', {'safe_zone': {'cooldown': 6}, 'health': {'health': 20}})
    ef = MaSurvivalVec(user, 70, seed=3, auto_reset='terminal', obs_layout='flat', global_state=True)
    ed = MaSurvivalVec(user, 70, seed=3, auto_reset='terminal')
    ef.reset(); od = ed.reset()
    _check_pieces('reset', ef, od)
    g = torch.Generator(device='cuda'); g.manual_seed(3)
    fin_total = 0
    for t in range(80):
        a = _actions(g, 70, ef.n_agents)
        rf, rd = ef.step(a), ed.step(a)
        _check_pieces(t, ef, rd[0])
        _check_pieces((t, 'terminal'), ef, rd[3]['terminal_observation'], 'terminal_global_state', rd[2])
        fin_total += int(rd[2].sum())
    assert fin_total > 0
    ef.close(); ed.close()


def test_state_has_no_lidar_columns():
    from masurvival import _lib
    from masurvival.envs import MaSurvivalVec
    for name in ('ffa', 'ffa_lidar'):
        env = MaSurvivalVec(parity.variant(name), 40, seed=1, global_state=True)
        env.reset()
        assert env.state().shape == (40, 399) == (40, _lib.global_state_dim(env._rec))
        assert not any('lidar' in k for k in env.state_layout())
        _layout_is_the_row(env)
        env.close()


def test_state_cuda_graph_step_and_reset_envs():
    """a CUDA graph of step + reset_envs on a state-on handle replays to the eager run's rows"""
    import torch
    from masurvival.envs import MaSurvivalVec
    N, T = 300, 30
    user = _user('ffa_lidar', {'safe_zone': {'cooldown': 6}, 'health': {'health': 15}})
    eg, ee = (MaSurvivalVec(user, N, seed=8, auto_reset=False, max_episode_steps=T, global_state=True) for _ in range(2))
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
        assert _equal_bits(eg.state(), ee.state()), t
    assert eg.get_state().tobytes() == ee.get_state().tobytes()
    eg.close(); ee.close()


def test_state_enable_refusals_and_idempotence():
    import torch
    from masurvival import _lib
    from masurvival.envs import MaSurvival, MaSurvivalVec
    env = MaSurvivalVec(parity.variant('2v2'), 64, seed=1)
    env.reset()
    with pytest.raises(RuntimeError):
        env.state()
    with pytest.raises(RuntimeError):
        env.state_layout()
    assert env.state_space.shape == (195,)
    a = torch.zeros((64, env.n_agents, 6), dtype=torch.uint8, device='cuda')
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        env.step(a)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        env.step(a)
        with pytest.raises(_lib.MasurvError):
            env._h.enable_global_state(torch.cuda.current_stream().cuda_stream)
    assert not env._h.has_tensor('global_state')
    graph.replay()
    torch.cuda.synchronize()
    env._h.enable_global_state(0)
    env.global_state = True
    p = env.state().data_ptr()
    first = env.state().clone()
    env._h.enable_global_state(0)
    torch.cuda.synchronize()
    assert env._h.tensor_info('global_state')[0] == p and _equal_bits(env.state(), first)
    obs = env.observe()
    _check_pieces('late enable', env, obs)
    env.close()
    assert _lib.load().msv_enable_global_state(None, None) == -1
    single = MaSurvival(parity.variant('2v2'), global_state=True)
    single.reset()
    s = single.state()
    assert isinstance(s, np.ndarray) and s.dtype == np.float32 and s.shape == (195,)
    single.close()


def test_state_two_devices():
    import torch
    from masurvival.envs import MaSurvivalVec
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two visible devices')
    user = _user('ffa', {'safe_zone': {'cooldown': 8}})
    envs = [MaSurvivalVec(user, 64, device=d, seed=6, global_state=True) for d in (0, 1)]
    for e in envs:
        with torch.cuda.device(e.device):
            e.reset()
    g = torch.Generator(device='cpu'); g.manual_seed(0)
    for t in range(20):
        a = torch.randint(0, 2, (64, envs[0].n_agents, 6), dtype=torch.uint8, generator=g)
        for e in envs:
            with torch.cuda.device(e.device):
                e.step(a.to(f'cuda:{e.device}'))
        torch.cuda.synchronize(0); torch.cuda.synchronize(1)
        assert _equal_bits(envs[0].state().cpu(), envs[1].state().cpu()), t
    for e in envs:
        e.close()
