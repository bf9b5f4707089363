"""The kernels off the benchmark's shapes: every agent count and capacity class in lock-step with the
oracle, the observation of injected states (msv_observe), a sweep of lidar fans on crafted scenes,
terminal-observation capture across classes and observation modes, and the tile hand-off in batches
that need several waves.  Every entry asserts the capacity class it runs in (G lanes per environment:
2, 4, 8 for classes 0, 1, 2), so a change to the class rule cannot silently move it."""
import math

import numpy as np
import pytest

import obs_cases as oc
import parity
from parity import make_config, random_actions

pytestmark = pytest.mark.gpu

PER_ENV = ('zone', 'heals', 'boxes', 'box_items')     # stored once per env, expanded to every observer


def _assert_clean(r):
    assert r['state_fail'] == 0 and r['obs_fail'] == 0, r['details']
    assert r['state_exact_mismatch'] == 0 and r['obs_exact_mismatch'] == 0, r['details']
    assert r['stats_gpu'] == r['stats_oracle']


def _lanes(plan):
    return plan['threads_per_block'] // plan['envs_per_block']


def _user(over, fast=True):
    return parity.apply_overrides(parity.variant('1v1'), oc._merge(oc.FAST if fast else {}, over))


# ------------------------------------------------------------------ B.1 lock-step matrix
@pytest.mark.parametrize('name,over,cls', [(m[0], m[2], m[3]) for m in oc.MATRIX], ids=[m[0] for m in oc.MATRIX])
def test_lockstep_matrix(name, over, cls):
    import gpu_lockstep
    from masurvival import _lib
    rec = oc.matrix_config(over, auto_reset=True)
    assert oc.plan_class(rec) == cls
    for n in (37, 45, 53, 59):                          # a ragged last tile
        h = _lib.Handle(rec, n, 0, 1, 0)
        plan = h.tile_plan(); h.close()
        if n % plan['envs_per_block']:
            break
    assert n % plan['envs_per_block'] and _lanes(plan) == oc.LANES[cls], plan
    r = gpu_lockstep.run('1v1', n, 150, verbose=False, **oc._merge(oc.FAST, over))
    _assert_clean(r)
    assert r['dones'] > 0 and r['overflow_events'] == 0, (r['dones'], r['overflow_events'])


# ------------------------------------------------------ B.2 observation of injected states
OBS_CASES = [(m[0], m[2], m[3]) for m in oc.MATRIX] + [('2v2', None, 1), ('ffa', None, 2)]


def _env_config(name, over, auto_reset):
    if over is None:
        return parity.variant(name), make_config(name, auto_reset=auto_reset)
    return _user(over), oc.matrix_config(over, auto_reset=auto_reset)


@pytest.mark.parametrize('name,over,cls', OBS_CASES, ids=[c[0] for c in OBS_CASES])
def test_observe_injected_states(name, over, cls):
    """msv_observe after msv_set_state against the oracle's set_state + observe, bit-exact on every key"""
    import pyoracle as po
    from masurvival.envs import MaSurvivalVec
    cfg, rec = _env_config(name, over, False)
    N = 43                                              # not a multiple of 32 (k_obs2 tile) nor of 2, 4, 8 (k_lidar EB)
    env = MaSurvivalVec(cfg, N, seed=5, auto_reset=False)
    assert _lanes(env.tile_plan()) == oc.LANES[cls] and oc.plan_class(rec) == cls
    env.reset()
    rng = np.random.default_rng(17)
    orcs = [po.OracleEnv(rec, seed=5, env_id=e) for e in range(N)]
    states, tags, want = [], [], []
    for e in range(N):
        orcs[e].reset()
        cases = oc.observation_states(rec, orcs[e].get_state(), rng)
        tag, s = cases[e % len(cases)]
        orcs[e].set_state(s)
        want.append(orcs[e].observe())
        states.append(s); tags.append(tag)
    assert len(set(tags)) == len(cases)                 # every kind of crafted state is in the batch
    env.set_state(np.array(states))
    env._h.observe()
    import torch
    torch.cuda.synchronize()
    keys = list(po.obs_dims(rec).keys())
    raw = {k: env._h.tensor(k).cpu().numpy() for k in keys}
    for e in range(N):
        for k in keys:
            g = raw[k][e]
            if k in PER_ENV:
                g = np.broadcast_to(g[None], (int(rec['n_agents']),) + g.shape)
            assert np.array_equal(g, want[e][k]), (name, tags[e], e, k)
    obs = env.observe()                                 # the public path returns the same tensors
    torch.cuda.synchronize()
    for k in keys:
        v = obs[k].cpu().numpy()
        for e in range(N):
            assert np.array_equal(v[e], want[e][k]), (name, tags[e], e, k)
    env.close()


# ------------------------------------------------------------------- B.3 lidar fan sweep
# (A, L, fov, depth): every value of every axis, every fov with two values of L, every A with a fan wider
# than pi.  k_lidar runs EB = 8 // A environments per block (A = 1: 8, 2: 4, 3: 2, 4: 2, 5: 1, 8: 1).
P = math.pi
FANS = [(1, 1, 0.1, 10.0), (2, 9, 0.1, 2.0), (3, 2, 0.8 * P, 0.4), (4, 32, 0.8 * P, 10.0), (5, 31, 2.85, 10.0),
        (8, 9, 2.85, 30.0), (1, 32, 2.95, 2.0), (2, 31, 2.95, 10.0), (3, 9, P, 10.0), (4, 1, P, 30.0),
        (1, 9, 3.2, 10.0), (5, 32, 3.2, 2.0), (2, 2, 1.5 * P, 10.0), (8, 31, 1.5 * P, 10.0), (3, 32, 2 * P, 30.0),
        (4, 9, 2 * P, 0.4), (5, 1, 1.5 * P, 10.0), (8, 32, 3.2, 0.4), (2, 32, 2 * P, 10.0), (1, 2, 2 * P, 2.0),
        (3, 31, 3.2, 2.0), (4, 2, 1.5 * P, 2.0)]


def test_lidar_fan_sweep():
    import torch
    import pyoracle as po
    from masurvival import _lib
    kinds, nonconvex, single, n_rays, n_good = set(), 0, 0, 0, 0
    for A, L, fov, depth in FANS:
        rec = oc.lidar_config(A, L, fov, depth)
        EB = max(1, 8 // A)
        o = po.OracleEnv(rec, seed=5, env_id=1)
        o.reset()
        rng = np.random.default_rng(A * 1000 + L)
        cases = oc.lidar_states(rec, o.get_state(), rng)
        if len(cases) % 2 == 0:
            cases.append(cases[0])                       # a ragged last k_lidar block
        N = len(cases)
        h = _lib.Handle(rec, N, 0, 5, 0)
        h.reset()
        h.set_state(np.array([s for _, s in cases]))
        h.observe()
        torch.cuda.synchronize()
        keys = list(po.obs_dims(rec).keys())
        g = {k: h.tensor(k).cpu().numpy() for k in keys}
        for e, (tag, s) in enumerate(cases):
            o.set_state(s)
            want = o.observe()
            for k in keys:
                v = np.broadcast_to(g[k][e][None], (A,) + g[k][e].shape) if k in PER_ENV else g[k][e]
                assert np.array_equal(v, want[k]), ((A, L, fov, depth), 'EB', EB, tag, k,
                                                    np.argwhere(v != want[k])[:4].tolist() if v.shape == want[k].shape else v.shape)
            f, hit, good = oc.lidar_reference(rec, s)
            alive = s['alive'][:A] != 0
            ok = good & alive[:, None]
            n_rays += int(alive.sum()) * L; n_good += int(ok.sum())
            assert np.array_equal(g['lidar_hit'][e][ok], hit[ok]), ((A, L, fov, depth), tag)
            assert np.all(np.abs(g['lidar_frac'][e][ok] - f[ok]) * depth <= 1e-4), ((A, L, fov, depth), tag)
            kinds |= {int(x) >> 8 for x in g['lidar_hit'][e][alive].ravel()}
        ang = oc.ray_angles(rec)
        nonconvex += L > 1 and 0.5 * (ang[-1] - ang[0]) >= 1.45
        single += L == 1
        h.close(); o.close()
    assert kinds >= {0, oc.KIND_AGENT, oc.KIND_BOX, oc.KIND_ITEM, oc.KIND_HEAL, oc.KIND_WALL}, kinds
    assert nonconvex >= 8 and single >= 3
    assert n_good >= 0.94 * n_rays, 'well-conditioned %d of %d rays (%.1f %% excluded)' % (n_good, n_rays, 100 - 100 * n_good / n_rays)


# ---------------------------------------------------------------- B.4 terminal capture
_M = dict((m[0], m[2]) for m in oc.MATRIX)
TERMINAL = [('1v1', None, 0, 97),
            ('2v2_partial', {'agents': {'n_agents': 4, 'agent_size': 1}, 'teams': {'twoteams': True}, 'observation': {'omniscent': False}}, 1, 98),
            ('ffa', None, 2, 35), ('a3_teams', _M['a3_teams'], 1, 39), ('a3_partial', _M['a3_partial'], 1, 43),
            ('a6_partial', _M['a6_partial'], 2, 38), ('exotic_b', {k: dict(v) for k, v in parity.EXOTIC_B.items()}, 0, 41),
            ('1v1_heal_only', None, 0, 66), ('a7_lidar', _M['a7_lidar'], 2, 35)]


@pytest.mark.parametrize('name,over,cls,N', TERMINAL, ids=[t[0] for t in TERMINAL])
def test_terminal_capture_matrix(name, over, cls, N):
    """auto_reset='terminal': the trajectory is bit-identical to auto_reset=True, and every terminal_<key>
    (lidar included) equals the observation the oracle, stepped without auto-reset, returns on the step
    its episode ends.  Episodes end with the last agent (team) standing, so the terminal row of a live
    observer is compared; the first episode starts with box items on the floor in front of the agents, so
    the partial-observability item masks and the lidar of a survivor see them."""
    import torch
    import pyoracle as po
    from masurvival.envs import MaSurvivalVec
    fast = {'safe_zone': {'cooldown': 6}, 'health': {'health': 10}, 'gameover': {'mode': 'lastalive'}}
    if over is None:
        cfg = parity.apply_overrides(parity.variant(name), fast)
        rec0 = make_config(name, auto_reset=False, **fast)
    else:
        cfg = parity.apply_overrides(parity.variant('1v1'), oc._merge(over, fast))
        rec0 = make_config('1v1', auto_reset=False, **oc._merge(over, fast))
    A, B = int(rec0['n_agents']), int(rec0['n_boxes'])
    partial, L = not rec0['omniscient'], int(rec0['lidar_n'])
    et = MaSurvivalVec(cfg, N, seed=9, auto_reset='terminal')
    e1 = MaSurvivalVec(cfg, N, seed=9, auto_reset=True)
    assert _lanes(et.tile_plan()) == oc.LANES[cls] and oc.plan_class(rec0) == cls
    orcs = [po.OracleEnv(rec0, seed=9, env_id=e) for e in range(N)]
    et.reset(); e1.reset()
    rng = np.random.default_rng(1)
    states = []
    for o in orcs:
        o.reset()
        states.append(oc.items_in_view(rec0, o.get_state(), rng))
        o.set_state(states[-1])
    et.set_state(np.array(states)); e1.set_state(np.array(states))
    keys = list(po.obs_dims(rec0))
    checked = live = items_seen = lidar_hits = 0
    for t in range(100):
        act = random_actions(rng, N, A)
        a = torch.as_tensor(act).cuda()
        snap = oc.terminal_snapshot(et._h)
        ot, rt, dt, info = et.step(a)
        oc.assert_unfinished_rows_kept(et._h, snap, dt, t)
        o1, r1, d1, _ = e1.step(a)
        for k in o1:
            assert torch.equal(ot[k], o1[k]), (t, k)
        assert torch.equal(rt, r1) and torch.equal(dt, d1)
        assert set(info['terminal_observation']) == set(keys)
        dn = dt.cpu().numpy()
        term = {k: v.cpu().numpy() for k, v in info['terminal_observation'].items()}
        for e in range(N):
            oo = orcs[e].step(act[e])
            assert bool(dn[e]) == oo['done'], (t, e)
            if oo['done']:
                for k in keys:
                    assert np.array_equal(term[k][e], oo[k]), (t, e, k)
                checked += 1
                live += int(np.any(oo['agent'][:, -7] > 0))               # an observer alive at the end (health column)
                if partial and B > 0:
                    items_seen += int(np.any(oo['box_items_mask'] == 0))  # an item on the floor that a live observer sees
                if L > 0:
                    lidar_hits += int(np.any(oo['lidar_hit'] != 0))
                orcs[e].reset()
    assert et.get_state().tobytes() == e1.get_state().tobytes()
    assert checked >= 5 and live >= checked // 2, (checked, live)
    if partial and B > 0:
        assert items_seen >= 3, items_seen
    if L > 0:
        assert lidar_hits >= 3, lidar_hits
    assert et._h.overflow_events() == 0
    et.close(); e1.close()


# ------------------------------------------------------------ B.5 multi-wave hand-off
def _multiwave_n(rec, sms):
    """a batch size whose tile plan needs about 1.5 waves of the largest tile, with a ragged last tile"""
    import ctypes
    from masurvival import _lib
    L = _lib.load()
    buf = np.array(rec, dtype=_lib.CONFIG_DT).reshape(1)
    out = (ctypes.c_int32 * 4)()
    _lib.check(L.msv_plan_tile(buf.ctypes.data, 1 << 24, sms, 227 * 1024, out))
    return (3 * sms // 2) * int(out[0]) + 13


@pytest.mark.parametrize('vname,steps', [('2v2', 120), ('ffa_lidar', 40), ('1v1', 150)])
def test_tile_hand_off_multi_wave(vname, steps, monkeypatch):
    import torch
    from masurvival.envs import MaSurvivalVec
    over = {'safe_zone': {'cooldown': 10}, 'health': {'health': 20}}
    cfg = parity.apply_overrides(parity.variant(vname), over)
    rec = make_config(vname, auto_reset=True, **over)
    A = int(rec['n_agents'])
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N = _multiwave_n(rec, sms)
    monkeypatch.delenv('MSV_NO_HANDOFF', raising=False)
    e1 = MaSurvivalVec(cfg, N, seed=11)
    monkeypatch.setenv('MSV_NO_HANDOFF', '1')
    e2 = MaSurvivalVec(cfg, N, seed=11)
    monkeypatch.delenv('MSV_NO_HANDOFF', raising=False)
    p1, p2 = e1.tile_plan(), e2.tile_plan()
    G = oc.LANES[oc.plan_class(rec)]
    assert p1['observation_hand_off'] and not p2['observation_hand_off']
    assert p1['threads_per_block'] == p1['envs_per_block'] * G and p1['blocks'] > sms, (p1, sms)
    assert N % p1['envs_per_block'] != 0
    g = torch.Generator(device='cuda'); g.manual_seed(2)
    dones = 0
    e1.reset(); e2.reset()
    for t in range(steps):
        a = torch.empty((N, A, 6), dtype=torch.uint8, device='cuda')
        a[..., :3] = torch.randint(0, 3, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
        a[..., 3:] = torch.randint(0, 2, (N, A, 3), dtype=torch.uint8, device='cuda', generator=g)
        o1, r1, d1, _ = e1.step(a)
        o2, r2, d2, _ = e2.step(a)
        if t % 7 == 0 or t == steps - 1:
            for k in o1:
                assert torch.equal(o1[k], o2[k]), (t, k)
            assert torch.equal(r1, r2) and torch.equal(d1, d2)
        dones += int(d1.sum())
    torch.cuda.synchronize()
    assert dones > 0
    assert e1.get_state().tobytes() == e2.get_state().tobytes()
    assert e1._h.overflow_events() == 0 and e2._h.overflow_events() == 0   # (includes the hand-off's give-up flag)
    e1.close(); e2.close()
