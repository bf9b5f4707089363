"""Episode control on the device: msv_reset_envs (reset the environments a mask selects) and the step limit
(msv_config.max_episode_steps), in lock-step with the CPU oracle.  The oracle has no step limit: the tests
apply the rule to it (truncated = steps >= T and not done) and reset its environments where the library
does."""
import ctypes

import numpy as np
import pytest

import obs_cases as oc
import parity
from parity import compare_obs, compare_states, random_actions

pytestmark = pytest.mark.gpu

DEDUP = ('zone', 'heals', 'boxes', 'box_items')      # stored once per env, expanded to the reference shape


def _user(name, over):
    return parity.apply_overrides(parity.variant(name), {k: dict(v) for k, v in over.items()})


def _names(h, keys):
    """every output tensor the handle has: observations, step outputs, terminal copies"""
    cand = keys + ['rewards', 'dones', 'truncated', 'episode_return', 'episode_length', 'immune', 'br_over', 'br_results']
    cand += ['terminal_' + k for k in keys]
    return [k for k in cand if h.has_tensor(k)]


def _snapshot(h, names):
    import torch
    torch.cuda.synchronize()
    return {k: h.tensor(k).cpu().numpy().copy() for k in names}


def _expand(k, arr, A):
    return np.broadcast_to(arr[None], (A,) + arr.shape) if k in DEDUP else arr


def _check_env(tag, e, sg, so, g, oo, keys, A, step_outputs=True):
    """state record and observation row of env e against the oracle (bit-exact)"""
    if sg[e].tobytes() != so.tobytes():
        raise AssertionError((tag, e, 'state', compare_states(sg[e], so)[0][:6]))
    og = {k: _expand(k, g[k][e], A) for k in keys}
    ref = {k: oo[k] for k in keys}
    if step_outputs:
        og['rewards'] = g['rewards'][e]; og['done'] = bool(g['dones'][e])
        ref['rewards'] = oo['rewards']; ref['done'] = oo['done']
    ex, _ = compare_obs(og, ref)
    assert not ex, (tag, e, 'obs', ex[:6])


# (id, user config, N): 2v2, ffa with lidar on a ragged last tile, partial observability, one matrix entry per
# capacity class (2, 4 and 8 lanes per environment)
MASK_CASES = [
    ('2v2', _user('2v2', {'safe_zone': {'cooldown': 8}, 'health': {'health': 30}}), 96),
    ('ffa_lidar', _user('ffa_lidar', {'safe_zone': {'cooldown': 6}, 'health': {'health': 20}}), 100),
    ('2v2_partial', _user('2v2', oc._merge(oc.PARTIAL, {'safe_zone': {'cooldown': 8}, 'health': {'health': 30}})), 64),
] + [(cid, _user('1v1', oc._merge(oc.FAST, over)), n)
     for (cid, _, over, cls), n in zip([m for m in oc.MATRIX if m[0] in ('a1_default', 'a3_teams', 'a7_lidar')], (70, 45, 30))]


@pytest.mark.parametrize('mode', [False, True, 'terminal'])
@pytest.mark.parametrize('cid,user,N', MASK_CASES, ids=[c[0] for c in MASK_CASES])
def test_masked_reset_lockstep(cid, user, N, mode):
    """random masks of about a quarter of the batch (one empty, one all-ones) between steps; the oracle resets the
    same envs.  State, observations, rewards and dones match every step; around every reset_envs the rows of the
    unmasked envs of every output tensor stay bit-identical; manual resets are not counted as episodes."""
    import torch
    import pyoracle as po
    from masurvival.envs import MaSurvivalVec
    seed = 13
    env = MaSurvivalVec(user, N, seed=seed, auto_reset=mode)
    rec, A = env._rec, env.n_agents
    orcs = [po.OracleEnv(rec, seed=seed, env_id=e) for e in range(N)]
    keys = list(po.obs_dims(rec).keys())
    names = _names(env._h, keys)
    env.reset()
    outs = [o.reset() for o in orcs]
    g, sg = _snapshot(env._h, names), env.get_state()
    for e in range(N):
        _check_env('reset', e, sg, orcs[e].get_state(), g, outs[e], keys, A)
    rng = np.random.default_rng(seed)
    n_resets = n_masks = 0
    for t in range(120):
        act = random_actions(rng, N, A)
        env.step(torch.as_tensor(act).cuda())
        outs = [orcs[e].step(act[e]) for e in range(N)]
        g, sg = _snapshot(env._h, names), env.get_state()
        for e in range(N):
            _check_env(f'step {t}', e, sg, orcs[e].get_state(), g, outs[e], keys, A)
            if outs[e]['done']:
                assert np.array_equal(g['episode_return'][e], outs[e]['episode_return']), (t, e)
                assert int(g['episode_length'][e]) == outs[e]['episode_length'], (t, e)
        if t % 5 != 3:
            continue
        mask = np.zeros(N, bool) if t == 8 else np.ones(N, bool) if t == 13 else rng.random(N) < 0.25
        form = n_masks % 3
        n_masks += 1
        if form == 0:
            arg = torch.as_tensor(mask).cuda()                               # device bool, used in place
        elif form == 1:
            arg = mask                                                       # host boolean array
        else:
            arg = [int(i) for i in np.flatnonzero(mask)]                     # env indices
        before = g
        env.reset_envs(arg)
        after = _snapshot(env._h, names)
        for k in names:
            assert np.array_equal(after[k][~mask], before[k][~mask]), (t, k, 'unmasked rows changed')
        for k in ('episode_return', 'episode_length'):                       # the last finished episode's record stays
            assert np.array_equal(after[k][mask], before[k][mask]), (t, k)
        if 'truncated' in names:
            assert not after['truncated'][mask].any()
        for e in np.flatnonzero(mask):
            outs[e] = orcs[e].reset()
            n_resets += 1
        sg = env.get_state()
        for e in range(N):
            _check_env(f'reset_envs {t}', e, sg, orcs[e].get_state(), after, outs[e], keys, A)
    assert n_resets > N                                                      # the all-ones mask alone is N
    st = env.flush_stats()
    assert st['episodes'] == sum(int(o.flush_stats()['episodes']) for o in orcs)   # manual resets are not episodes
    env.close()


@pytest.mark.parametrize('mode,T', [(True, 0), ('terminal', 0), (False, 25)])
def test_all_ones_mask_equals_reset(mode, T):
    import torch
    from masurvival.envs import MaSurvivalVec
    N = 200
    user = _user('ffa_lidar', {'safe_zone': {'cooldown': 6}, 'health': {'health': 20}})
    e1, e2 = (MaSurvivalVec(user, N, seed=3, auto_reset=mode, max_episode_steps=T) for _ in range(2))
    names = _names(e1._h, list(e1.obs_shapes()))
    rng = np.random.default_rng(2)
    e1.reset(); e2.reset()
    for phase in range(2):
        for t in range(40):
            a = torch.as_tensor(random_actions(rng, N, 8)).cuda()
            e1.step(a); e2.step(a)
        e1.reset()
        if phase == 0:
            e2.reset_envs(torch.ones(N, dtype=torch.uint8, device='cuda'))
        else:
            e2.reset(options={'reset_mask': np.ones(N, bool)})
        s1, s2 = _snapshot(e1._h, names), _snapshot(e2._h, names)
        for k in names:
            assert np.array_equal(s1[k], s2[k]), (phase, k)
        assert e1.get_state().tobytes() == e2.get_state().tobytes()
    e1.close(); e2.close()


def test_hand_off_after_reset_envs(monkeypatch):
    """steps after masked resets: the tile hand-off gives what plain stream-ordered launches give"""
    import torch
    from masurvival.envs import MaSurvivalVec
    N, A = 1030, 4
    user = _user('2v2', {'safe_zone': {'cooldown': 10}, 'health': {'health': 20}})
    monkeypatch.delenv('MSV_NO_HANDOFF', raising=False)
    e1 = MaSurvivalVec(user, N, seed=11)
    monkeypatch.setenv('MSV_NO_HANDOFF', '1')
    e2 = MaSurvivalVec(user, N, seed=11)
    monkeypatch.delenv('MSV_NO_HANDOFF', raising=False)
    assert e1.tile_plan()['observation_hand_off'] and not e2.tile_plan()['observation_hand_off']
    g = torch.Generator(device='cuda'); g.manual_seed(4)
    e1.reset(); e2.reset()
    for t in range(80):
        a = torch.empty((N, A, 6), dtype=torch.uint8, device='cuda')
        a[..., :3] = torch.randint(0, 3, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
        a[..., 3:] = torch.randint(0, 2, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
        o1, r1, d1, _ = e1.step(a)
        o2, r2, d2, _ = e2.step(a)
        for k in o1:
            assert torch.equal(o1[k], o2[k]), (t, k)
        assert torch.equal(r1, r2) and torch.equal(d1, d2)
        if t % 4 == 1:
            m = torch.rand(N, device='cuda', generator=g) < 0.2
            o1 = e1.reset_envs(m); o2 = e2.reset_envs(m)
            for k in o1:
                assert torch.equal(o1[k], o2[k]), (t, k)
    assert e1.get_state().tobytes() == e2.get_state().tobytes()
    assert e1._h.overflow_events() == 0 and e2._h.overflow_events() == 0
    e1.close(); e2.close()


@pytest.mark.parametrize('T', [0, 30])
def test_cuda_graph_step_and_reset_envs(T):
    """a CUDA graph of step + reset_envs(mask computed on the device from dones), replayed, equals the eager run"""
    import torch
    from masurvival.envs import MaSurvivalVec
    N, A = 300, 4
    user = _user('2v2', {'safe_zone': {'cooldown': 6}, 'health': {'health': 15}})
    eg, ee = (MaSurvivalVec(user, N, seed=8, auto_reset=False, max_episode_steps=T) for _ in range(2))
    rng = np.random.default_rng(5)
    a_static = torch.zeros((N, A, 6), dtype=torch.uint8, device='cuda')

    def body(env):
        _, _, d, info = env.step(a_static)
        m = d.clone()
        if T:
            m |= info['truncated']
        env.reset_envs(m)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eg.reset(); ee.reset()
        for _ in range(3):                                 # warm-up (kernel attributes, side stream, tensor views)
            a_static.copy_(torch.as_tensor(random_actions(rng, N, A)))
            body(eg); body(ee)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body(eg)
    names = _names(eg._h, list(eg.obs_shapes()))
    resets = 0
    for t in range(60):
        a_static.copy_(torch.as_tensor(random_actions(rng, N, A)))
        graph.replay()
        body(ee)
        torch.cuda.synchronize()
        sg, se = _snapshot(eg._h, names), _snapshot(ee._h, names)
        for k in names:
            assert np.array_equal(sg[k], se[k]), (t, k)
        resets += int(ee.get_state()['steps'].tolist().count(0))
    assert eg.get_state().tobytes() == ee.get_state().tobytes()
    assert resets > 0
    eg.close(); ee.close()


def test_refusals_and_index_form():
    import torch
    from masurvival import _lib
    from masurvival.envs import MaSurvivalVec
    L = _lib.load()
    N = 64
    user = _user('2v2', {})
    e1, e2 = (MaSurvivalVec(user, N, seed=2, auto_reset=True) for _ in range(2))
    e1.reset(); e2.reset()
    n0 = e1.kernel_launches()
    assert L.msv_reset_envs(e1._h.h, None, None) == -1
    assert L.msv_reset_envs(None, ctypes.c_void_p(e1._h.tensor('dones').data_ptr()), None) == -1
    assert e1.kernel_launches() == n0
    bad = [torch.ones(N - 1, dtype=torch.uint8, device='cuda'), torch.ones(N, dtype=torch.float32, device='cuda'),
           torch.ones(N, dtype=torch.int64, device='cuda'), np.ones(N + 1, bool), [0, N], [-1], np.ones(N, np.float32)]
    if torch.cuda.device_count() > 1:
        bad.append(torch.ones(N, dtype=torch.uint8, device='cuda:1'))
    for m in bad:
        with pytest.raises(ValueError):
            e1.reset_envs(m)
    assert e1.kernel_launches() == n0
    rng = np.random.default_rng(1)
    for t in range(20):
        a = torch.as_tensor(random_actions(rng, N, 4)).cuda()
        e1.step(a); e2.step(a)
    idx = [3, 7, 11, 63]
    mask = torch.zeros(N, dtype=torch.bool, device='cuda'); mask[idx] = True
    o1 = e1.reset_envs(idx); o2 = e2.reset_envs(mask)
    for k in o1:
        assert torch.equal(o1[k], o2[k]), k
    assert e1.get_state().tobytes() == e2.get_state().tobytes()
    assert e1.kernel_launches() == e2.kernel_launches()               # the same launches either way, none for the refusals
    e1.close(); e2.close()


@pytest.mark.parametrize('mode', [True, 'terminal', False])
@pytest.mark.parametrize('T', [1, 37])
@pytest.mark.parametrize('name,N', [('2v2', 48), ('ffa_lidar', 24)])
def test_step_limit_lockstep(name, N, T, mode):
    import torch
    import pyoracle as po
    from masurvival.envs import MaSurvivalVec
    over = {'safe_zone': {'cooldown': 6}, 'health': {'health': 60}}
    seed = 5
    env = MaSurvivalVec(_user(name, over), N, seed=seed, auto_reset=mode, max_episode_steps=T)
    assert not env.tile_plan()['observation_hand_off']
    rec0 = parity.make_config(name, auto_reset=False, **over)                # the oracle never resets by itself
    A = env.n_agents
    orcs = [po.OracleEnv(rec0, seed=seed, env_id=e) for e in range(N)]
    keys = list(po.obs_dims(rec0).keys())
    names = _names(env._h, keys)
    assert 'truncated' in names
    env.reset()
    for o in orcs:
        o.reset()
    auto = mode is not False
    episodes = np.zeros(N, np.int64)
    n_done = n_trunc = 0
    rng = np.random.default_rng(seed)
    for t in range(80):
        act = random_actions(rng, N, A)
        before = oc.terminal_snapshot(env._h) if mode == 'terminal' else None
        _, _, d, info = env.step(torch.as_tensor(act).cuda())
        if before is not None:
            oc.assert_unfinished_rows_kept(env._h, before, d | info['truncated'], t)
        g, sg = _snapshot(env._h, names), env.get_state()
        tr = info['truncated'].cpu().numpy()
        term = {k: v.cpu().numpy() for k, v in info['terminal_observation'].items()} if mode == 'terminal' else None
        finished = []
        for e in range(N):
            oo = orcs[e].step(act[e])
            so = orcs[e].get_state()
            done, trunc = oo['done'], int(so['steps']) >= T and not oo['done']
            assert bool(g['dones'][e]) == done and bool(tr[e]) == trunc, (t, e)
            assert np.array_equal(g['rewards'][e], oo['rewards']), (t, e)
            if done or trunc:
                n_done += done; n_trunc += trunc
                ret, length = (oo['episode_return'], oo['episode_length']) if done else (so['ep_return'][:A], int(so['steps']))
                assert np.array_equal(g['episode_return'][e], ret) and int(g['episode_length'][e]) == length, (t, e)
                if term is not None:                                         # the episode's last observation, lidar included
                    for k in keys:
                        assert np.array_equal(term[k][e], oo[k]), (t, e, k)
                finished.append(e)
            if auto and (done or trunc):
                oo = orcs[e].reset()                                         # the library's auto-reset episode
                episodes[e] += 1
            so = orcs[e].get_state()
            so['stat_episodes'] = episodes[e]
            _check_env(f'step {t}', e, sg, so, g, oo, keys, A, step_outputs=False)
        if not auto and finished:                                            # the caller restarts them
            env.reset_envs(d | info['truncated'])
            g, sg = _snapshot(env._h, names), env.get_state()
            for e in finished:
                oo = orcs[e].reset()
                _check_env(f'reset_envs {t}', e, sg, orcs[e].get_state(), g, oo, keys, A)
            assert not g['truncated'][:N].any() and not g['dones'][finished].any()
    assert n_trunc > 0
    assert env.flush_stats()['episodes'] == (n_done + n_trunc if auto else 0)
    env.close()


@pytest.mark.parametrize('mode,launches', [(True, 3), (False, 2), ('terminal', 5)])
def test_unreached_limit_changes_nothing(mode, launches):
    """T = 10**6 is never reached: state and outputs equal a T = 0 handle that runs with the tile hand-off, and
    truncated stays zero.  The T = 0 handle launches what the parent commit launched per step."""
    import torch
    from masurvival.envs import MaSurvivalVec
    N, A = 500, 4
    user = _user('2v2', {'safe_zone': {'cooldown': 8}, 'health': {'health': 20}})
    e0 = MaSurvivalVec(user, N, seed=6, auto_reset=mode)
    e1 = MaSurvivalVec(user, N, seed=6, auto_reset=mode, max_episode_steps=10 ** 6)
    assert e0.tile_plan()['observation_hand_off'] == (mode != 'terminal') and not e1.tile_plan()['observation_hand_off']
    names = _names(e0._h, list(e0.obs_shapes()))
    e0.reset(); e1.reset()
    g = torch.Generator(device='cuda'); g.manual_seed(6)
    dones = 0
    for t in range(150):
        a = torch.empty((N, A, 6), dtype=torch.uint8, device='cuda')
        a[..., :3] = torch.randint(0, 3, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
        a[..., 3:] = torch.randint(0, 2, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
        n0 = e0.kernel_launches()
        _, _, d0, _ = e0.step(a)
        _, _, _, info = e1.step(a)
        assert e0.kernel_launches() - n0 == launches
        assert not bool(info['truncated'].any())
        s0, s1 = _snapshot(e0._h, names), _snapshot(e1._h, names)
        for k in names:
            assert np.array_equal(s0[k], s1[k]), (t, k)
        dones += int(d0.sum())
    assert dones > 0
    assert e0.get_state().tobytes() == e1.get_state().tobytes()
    assert e0.flush_stats() == e1.flush_stats()
    e0.close(); e1.close()


def test_host_forms_under_a_limit():
    import torch
    from masurvival.envs import MaSurvivalVec
    N, A = 300, 4
    user = _user('2v2', {'safe_zone': {'cooldown': 8}, 'health': {'health': 40}})
    e1, e2 = (MaSurvivalVec(user, N, seed=4, max_episode_steps=20) for _ in range(2))
    e1.reset(); e2.reset()
    rew = torch.empty((N, A), dtype=torch.float32).pin_memory()
    done = torch.empty((N,), dtype=torch.uint8).pin_memory()
    rng = np.random.default_rng(3)
    truncs = 0
    for t in range(50):
        a = random_actions(rng, N, A)
        _, r1, d1, info = e1.step(torch.as_tensor(a).cuda())
        if t % 2:
            rh, dh = e2.step_host(a)
        else:
            e2.step_host_async(a, rew, done); e2.step_host_wait()
            rh, dh = rew.numpy(), done.numpy()
        torch.cuda.synchronize()
        assert np.array_equal(r1.cpu().numpy(), rh) and np.array_equal(d1.cpu().numpy(), dh.astype(bool)), t
        assert torch.equal(info['truncated'], e2._h.tensor('truncated').view(torch.bool)), t
        truncs += int(info['truncated'].sum())
    assert truncs > 0
    assert e1.get_state().tobytes() == e2.get_state().tobytes()
    e1.close(); e2.close()
