"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU
oracle on identical seeded inputs.  Discrete outputs (health, inventories,
alive/done flags, masks, rewards, lidar hit ids, contact bookkeeping) must be
bit-exact; continuous outputs within 1e-4 relative (BASELINE.json north_star).
In practice every field is bit-exact and the tests also assert that."""
import math

import numpy as np
import pytest

import obs_cases as oc
import parity
from parity import compare_obs, compare_states, make_config, random_actions, scramble_state

pytestmark = pytest.mark.gpu

# every output tensor of a step besides the terminal-mode copies
OUTPUTS = oc.OBS_KEYS + ('lidar_frac', 'lidar_hit', 'rewards', 'dones', 'episode_return', 'episode_length', 'immune',
                         'br_over', 'br_results', 'truncated')


def _assert_clean(r, need_exact=True):
    assert r['state_fail'] == 0 and r['obs_fail'] == 0, r['details']
    if need_exact:
        assert r['state_exact_mismatch'] == 0 and r['obs_exact_mismatch'] == 0, r['details']
    assert r['stats_gpu'] == r['stats_oracle']


@pytest.mark.parametrize('variant,n,steps', [('2v2', 64, 150), ('1v1', 64, 150), ('1v1_heal_only', 64, 100),
                                             ('ffa', 16, 80), ('ffa_lidar', 8, 40)])
def test_lockstep_rollout(variant, n, steps):
    import gpu_lockstep
    r = gpu_lockstep.run(variant, n, steps, verbose=False)
    _assert_clean(r)


@pytest.mark.parametrize('variant,n,epb,steps', [('2v2', 224, 112, 130), ('ffa', 112, 56, 60), ('1v1', 512, 160, 100)])
def test_lockstep_production_tiles(variant, n, epb, steps, monkeypatch):
    """the tile shapes the planner picks for the BASELINE batch sizes (one block of up to 512 threads per SM:
    112 envs x 4 lanes, 56 x 8, and the largest 2-lane tile), in lock-step with the oracle"""
    import gpu_lockstep
    from masurvival import _lib
    monkeypatch.setenv('MSV_EPB', str(epb))
    h = _lib.Handle(make_config(variant, auto_reset=True), n, device=0, seed=1, env_offset=0)
    plan = h.tile_plan(); h.close()
    assert plan['envs_per_block'] == epb and plan['threads_per_block'] in (448, 320)
    r = gpu_lockstep.run(variant, n, steps, verbose=False, safe_zone={'cooldown': 15}, health={'health': 25})
    _assert_clean(r)
    assert r['dones'] > 0 and r['overflow_events'] == 0


def test_lockstep_fast_zone_and_resets():
    """short safe-zone phases: every env runs through shrink, endgame, death,
    death-drop and in-kernel auto-reset several times"""
    import gpu_lockstep
    r = gpu_lockstep.run('2v2', 48, 260, verbose=False, safe_zone={'cooldown': 8}, health={'health': 12})
    _assert_clean(r)
    assert r['dones'] > 40


def test_lockstep_partial_observability():
    """non-omniscient masks (env:706-739): Cameras over every body, Q1 row remap"""
    import gpu_lockstep
    r = gpu_lockstep.run('2v2', 48, 200, verbose=False, observation={'omniscent': False}, safe_zone={'cooldown': 20}, health={'health': 30})
    _assert_clean(r)
    r = gpu_lockstep.run('ffa', 12, 60, verbose=False, observation={'omniscent': False})
    _assert_clean(r)


def test_lockstep_exotic_configs():
    """configs far from the defaults (agent size, room size, fixed zone centres, 3 agents,
    2 inventory slots, lastalive, kill rewards, no heals, ownership without teams)"""
    import gpu_lockstep
    r = gpu_lockstep.run('1v1', 48, 200, verbose=False, **{k: dict(v) for k, v in parity.EXOTIC_A.items()})
    _assert_clean(r)
    assert r['dones'] > 10
    r = gpu_lockstep.run('1v1', 48, 150, verbose=False, **{k: dict(v) for k, v in parity.EXOTIC_B.items()})
    _assert_clean(r)


def test_lockstep_ownership():
    import gpu_lockstep
    r = gpu_lockstep.run('2v2', 32, 120, verbose=False, boxes={'ownership': True}, p_attack=0.9)
    _assert_clean(r)


def _scenario(variant, n, steps, seed, **over):
    """dense-interaction scenario: scrambled states injected on both sides"""
    import torch
    import pyoracle as po
    from masurvival import _lib
    rec = make_config(variant, auto_reset=False, **over)
    A = int(rec['n_agents'])
    h = _lib.Handle(rec, n, 0, seed, 0)
    orcs = [po.OracleEnv(rec, seed=seed, env_id=e) for e in range(n)]
    h.reset()
    rng = np.random.default_rng(seed)
    states = []
    for e in range(n):
        orcs[e].reset()
        s = scramble_state(orcs[e].get_state(), rec, rng)
        orcs[e].set_state(s)
        states.append(s)
    h.set_state(np.array(states))
    keys = list(po.obs_dims(rec).keys())
    bad = []
    events = {'toi': 0, 'deaths': 0, 'pick': 0}
    for t in range(steps):
        act = random_actions(rng, n, A, 0.6, 0.5, 0.3)
        a_dev = torch.as_tensor(act).cuda()
        h.step(a_dev.data_ptr())
        torch.cuda.synchronize()
        sg = h.get_state()
        g = {k: h.tensor(k).cpu().numpy() for k in keys + ['rewards', 'dones']}
        for e in range(n):
            oo = orcs[e].step(act[e])
            events['toi'] += oo['n_toi_events']
            so = orcs[e].get_state()
            ex, fl = compare_states(sg[e], so)
            og = {k: (np.broadcast_to(g[k][e][None], (A,) + g[k][e].shape) if k in ('zone', 'heals', 'boxes', 'box_items') else g[k][e]) for k in keys}
            og['rewards'] = g['rewards'][e]; og['done'] = bool(g['dones'][e])
            oex, ofl = compare_obs(og, oo)
            if ex or oex:
                bad.append((t, e, ex[:4], oex[:4]))
                h.set_state(np.array([so]), first=e)
            events['deaths'] += int((so['alive'][:A] == 0).sum())
            events['pick'] += int(so['inv_n'][:A].sum())
    assert h.overflow_events() == 0
    h.close()
    return bad, events


@pytest.mark.parametrize('variant,n,steps,over', [
    ('2v2', 96, 40, {}), ('1v1', 96, 40, {}), ('ffa', 24, 30, {}),
    ('2v2', 64, 40, {'boxes': {'ownership': True}}),
    ('2v2', 64, 40, {'observation': {'omniscent': False}}),
])
def test_scrambled_scenarios(variant, n, steps, over):
    bad, events = _scenario(variant, n, steps, seed=11, **over)
    assert not bad, bad[:5]
    assert events['toi'] > 0


def test_step_host_matches_step_and_dlpack_views():
    """msv_step_host (host buffers) and msv_step (device buffer) are the same
    computation; DLPack views alias library memory with reference shapes."""
    import torch
    from masurvival.envs import MaSurvivalVec
    from masurvival.config import variant
    N = 256
    e1 = MaSurvivalVec(variant('2v2'), N, seed=3)
    e2 = MaSurvivalVec(variant('2v2'), N, seed=3)
    o1 = e1.reset(); e2.reset()
    assert o1['agent'].shape == (N, 4, 9) and o1['zone'].shape == (N, 4, 6)
    assert o1['boxes'].shape == (N, 4, 4, 11) and o1['boxes'].stride(1) == 0
    assert o1['others'].shape == (N, 4, 3, 9) and o1['heal_slot'].shape == (N, 4, 1, 1)
    rng = np.random.default_rng(0)
    for t in range(30):
        a = random_actions(rng, N, 4)
        obs, rew, done, info = e1.step(torch.as_tensor(a).cuda())
        rh, dh = e2.step_host(a)
        torch.cuda.synchronize()
        assert np.array_equal(rew.cpu().numpy(), rh) and np.array_equal(done.cpu().numpy().astype(np.uint8), dh)
    s1, s2 = e1.get_state(), e2.get_state()
    assert s1.tobytes() == s2.tobytes()
    p = obs['agent'].data_ptr()
    obs2, *_ = e1.step(torch.as_tensor(a).cuda())
    assert obs2['agent'].data_ptr() == p  # zero-copy: same HBM every step
    e1.close(); e2.close()


def test_full_size_properties():
    """BASELINE size (16384 envs): determinism and domain invariants."""
    import torch
    from masurvival.envs import MaSurvivalVec
    from masurvival.config import variant
    N = 16384
    envs = [MaSurvivalVec(variant('2v2'), N, seed=5) for _ in range(2)]
    for e in envs:
        e.reset()
    g = torch.Generator(device='cuda'); g.manual_seed(0)
    tot_done = 0
    for t in range(120):
        a = torch.empty((N, 4, 6), dtype=torch.uint8, device='cuda')
        a[..., :3] = torch.randint(0, 3, (N, 4, 3), dtype=torch.uint8, device='cuda', generator=g)
        a[..., 3:] = torch.randint(0, 2, (N, 4, 3), dtype=torch.uint8, device='cuda', generator=g)
        outs = [e.step(a) for e in envs]
        tot_done += int(outs[0][2].sum())
    o0, r0, d0, _ = outs[0]; o1, r1, d1, _ = outs[1]
    for k in o0:
        assert torch.equal(o0[k], o1[k]), k          # same seed + actions -> identical (no atomics, no races)
    assert torch.equal(r0, r1) and torch.equal(d0, d1)
    ag = o0['agent']
    assert torch.all(ag[..., 3:5].abs() <= 10.0)      # nobody tunnels through the walls (TOI)
    hp = ag[..., 2]
    assert torch.all(hp == hp.round()) and torch.all(hp >= 0)
    assert torch.all((o0['others_mask'] == 0) | (o0['others_mask'] == 1))
    assert torch.all((r0 == 1) | (r0 == -1))
    st = envs[0].flush_stats()
    assert st['steps'] == N * 120 and st['episodes'] == tot_done
    assert envs[0]._h.overflow_events() == 0      # no fixed-capacity list ever overflowed
    for e in envs:
        e.close()


@pytest.mark.parametrize('vname,N,steps', [('2v2', 4100, 260), ('ffa_lidar', 1030, 60)])
def test_tile_hand_off_equals_plain_launches(vname, N, steps, monkeypatch):
    """The observation kernel consumes k_step's tiles in the order they finish (completion queue +
    programmatic dependent launch, k_step itself dependent on the previous step's observation kernel).
    The outputs must be bit-identical to plain stream-ordered launches, on a ragged batch (padding
    environments in the last tile), on a stream of our own, with episode ends and in-kernel resets."""
    import torch
    from masurvival.envs import MaSurvivalVec
    from masurvival.config import variant
    A = 4 if vname == '2v2' else 8
    over = {'safe_zone': {'cooldown': 10}, 'health': {'health': 20}}
    cfg = parity.apply_overrides(variant(vname), over)
    monkeypatch.delenv('MSV_NO_HANDOFF', raising=False)
    e1 = MaSurvivalVec(cfg, N, seed=11)
    monkeypatch.setenv('MSV_NO_HANDOFF', '1')
    e2 = MaSurvivalVec(cfg, N, seed=11)
    monkeypatch.delenv('MSV_NO_HANDOFF', raising=False)
    p1, p2 = e1._h.tile_plan(), e2._h.tile_plan()
    assert p1['observation_hand_off'] and not p2['observation_hand_off']
    assert p1['envs_per_block'] * p1['blocks'] >= N and p1['threads_per_block'] <= 512
    assert p1['blocks'] <= 148 or p1['threads_per_block'] == 512    # one wave of one block per SM, else full tiles
    g = torch.Generator(device='cuda'); g.manual_seed(2)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        o1 = e1.reset(); o2 = e2.reset()
        dones = 0
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
    st.synchronize()
    assert dones > N // 4
    assert e1.get_state().tobytes() == e2.get_state().tobytes()
    assert e1._h.overflow_events() == 0 and e2._h.overflow_events() == 0   # (includes the hand-off's own fault flag)
    e1.close(); e2.close()


def test_golden_fixtures_on_gpu():
    """the committed golden vectors (recorded from the reference's own Python,
    tests/golden/make_golden.py) replayed through the C ABI on the GPU"""
    import torch
    import test_cpu_golden as tg
    from masurvival import _lib
    import pyoracle as po
    for path in tg.GOLDEN:
        g = np.load(path)
        rec = tg.case_config(path)
        A = int(rec['n_agents'])
        seed, env_id, _ = [int(v) for v in g['meta']]
        h = _lib.Handle(rec, 1, 0, seed, env_id)
        keys = list(po.obs_dims(rec).keys())
        for r in range(len(g['kind'])):
            if g['kind'][r] == 0:
                h.reset()
            else:
                a = torch.as_tensor(g['actions'][r][None]).cuda()
                h.step(a.data_ptr())
            torch.cuda.synchronize()
            for k in keys + list(tg.EXTRA_KEYS):
                if k not in g.files:
                    continue
                v = h.tensor(k).cpu().numpy()[0]
                if k in ('zone', 'heals', 'boxes', 'box_items'):
                    v = np.broadcast_to(v[None], (A,) + v.shape)
                assert np.array_equal(v, g[k][r]), (path, r, k)
            if g['kind'][r] == 1:
                assert np.array_equal(h.tensor('rewards').cpu().numpy()[0], g['rewards'][r]), (path, r)
                assert bool(h.tensor('dones').cpu().numpy()[0]) == bool(g['done'][r]), (path, r)
        h.close()


def test_terminal_observation_capture():
    """auto_reset='terminal': same trajectory as the in-kernel reset, and the finished episode's
    last observation equals the observation the ORACLE (stepped without auto-reset) returns on the
    step its episode ends"""
    import torch
    import pyoracle as po
    from masurvival.envs import MaSurvivalVec
    N = 96
    over = {'safe_zone': {'cooldown': 6}, 'health': {'health': 10}}
    cfg = parity.apply_overrides(parity.variant('2v2'), over)
    rec0 = make_config('2v2', auto_reset=False, **over)
    et = MaSurvivalVec(cfg, N, seed=9, auto_reset='terminal')
    e1 = MaSurvivalVec(cfg, N, seed=9, auto_reset=True)
    orcs = [po.OracleEnv(rec0, seed=9, env_id=e) for e in range(N)]
    et.reset(); e1.reset()
    for o in orcs:
        o.reset()
    keys = [k for k in po.obs_dims(rec0)]
    rng = np.random.default_rng(1)
    checked = 0
    for t in range(90):
        act = random_actions(rng, N, 4)
        a = torch.as_tensor(act).cuda()
        ot, rt, dt, info = et.step(a)
        o1, r1, d1, _ = e1.step(a)
        for k in o1:
            assert torch.equal(ot[k], o1[k]), k
        assert torch.equal(rt, r1) and torch.equal(dt, d1)
        dn = dt.cpu().numpy()
        term = {k: v.cpu().numpy() for k, v in info['terminal_observation'].items()}
        for e in range(N):
            oo = orcs[e].step(act[e])
            assert bool(dn[e]) == oo['done'], (t, e)
            if oo['done']:
                for k in keys:
                    assert np.array_equal(term[k][e], oo[k]), (t, e, k)     # the oracle's last observation of the episode
                checked += 1
                orcs[e].reset()                                             # oracle episode n+1 == the GPU's auto-reset episode
    assert et.get_state().tobytes() == e1.get_state().tobytes()
    assert checked > 60
    et.close(); e1.close()


def test_abi_tensor_info_errors_and_lifetime():
    """msv_tensor_info shapes/strides/dtypes, unknown names, byte accounting, state round trip"""
    import ctypes
    import torch
    from masurvival import _lib
    rec = make_config('ffa_lidar', auto_reset=True)
    h = _lib.Handle(rec, 100, 0, 1, 0)                 # 100 is not a multiple of the 64-env block
    L = _lib.load()
    h.reset()
    ptr, nd, dt = ctypes.c_void_p(), ctypes.c_int32(), ctypes.c_int32()
    shape, strides = (ctypes.c_int64 * 4)(), (ctypes.c_int64 * 4)()
    rc = L.msv_tensor_info(h.h, b'others', ctypes.byref(ptr), ctypes.byref(nd), shape, strides, ctypes.byref(dt))
    assert rc == 0 and nd.value == 4 and list(shape) == [100, 8, 7, 8] and list(strides) == [448, 56, 8, 1] and dt.value == 0
    assert L.msv_tensor_info(h.h, b'lidar_hit', ctypes.byref(ptr), ctypes.byref(nd), shape, strides, ctypes.byref(dt)) == 0 and dt.value == 2
    assert L.msv_tensor_info(h.h, b'dones', ctypes.byref(ptr), ctypes.byref(nd), shape, strides, ctypes.byref(dt)) == 0 and dt.value == 1 and list(shape)[:1] == [100]
    assert L.msv_tensor_info(h.h, b'nope', None, None, None, None, None) == -4      # MSV_ERR_NAME
    assert b'nope' in L.msv_last_error(h.h)
    t = h.tensor('agent')
    assert t.shape == (100, 8, 8) and t.is_cuda and t.data_ptr() == h.tensor('agent').data_ptr()
    assert h.tensor('lidar_hit').dtype == torch.int32 and h.tensor('dones').dtype == torch.uint8
    assert h.bytes_per_env_step() > h.obs_bytes_per_env() > 0
    assert h.obs_bytes_per_env() == 4 * _stored_obs_floats(h)
    # checkpoint / resume: get_state -> set_state is the identity, and a restored env continues identically
    a = torch.zeros((100, 8, 6), dtype=torch.uint8, device='cuda'); a[..., :3] = 2; a[..., 3] = 1
    for _ in range(25):
        h.step(a.data_ptr())
    snap = h.get_state()
    for _ in range(10):
        h.step(a.data_ptr())
    torch.cuda.synchronize()
    ref_obs = h.tensor('agent').clone(); ref_state = h.get_state()
    h.set_state(snap)
    assert h.get_state().tobytes() == snap.tobytes()
    for _ in range(10):
        h.step(a.data_ptr())
    torch.cuda.synchronize()
    assert torch.equal(h.tensor('agent'), ref_obs) and h.get_state().tobytes() == ref_state.tobytes()
    assert h.get_state(first=99, count=1).shape == (1,)
    with pytest.raises(_lib.MasurvError):
        h.get_state(first=100, count=1)
    h.close()
    # the observation bytes per env are the stored observation tensors, for every agent count, class, H = 0 and B = 0
    recs = [oc.matrix_config(m[2]) for m in oc.MATRIX] + [make_config(n) for n in ('2v2', 'ffa', '1v1_heal_only')]
    recs.append(make_config('1v1', **{k: dict(v) for k, v in parity.EXOTIC_B.items()}))
    for rec in recs:
        h = _lib.Handle(rec, 37, 0, 1, 0)
        assert h.obs_bytes_per_env() == 4 * _stored_obs_floats(h), rec
        h.close()


def _stored_obs_floats(h):
    """floats per environment of the observation tensors as msv_tensor_info shapes them (zone, heals, boxes and
    box_items are stored once per env; a key the config does not have counts 0)"""
    import ctypes
    from masurvival import _lib
    nd, shape, n = ctypes.c_int32(), (ctypes.c_int64 * 4)(), 0
    for k in oc.OBS_KEYS:
        if _lib.load().msv_tensor_info(h.h, k.encode(), None, ctypes.byref(nd), shape, None, None) == 0:
            n += math.prod(shape[1:nd.value])
    return n


def test_two_devices_in_one_process():
    """The same ffa batch (8-lane class: the largest observation stage) on device 0 and device 1 of one process,
    stepped with the same actions, gives the same outputs: each handle prepares its kernels on its own device."""
    import torch
    from masurvival import _lib
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two visible devices')
    rec = make_config('ffa', auto_reset=True)
    N, A = 100, int(rec['n_agents'])
    hs = [_lib.Handle(rec, N, d, 3, 0) for d in (0, 1)]
    assert [h.tile_plan()['threads_per_block'] // h.tile_plan()['envs_per_block'] for h in hs] == [8, 8]
    names = [n for n in OUTPUTS if hs[0].has_tensor(n)]
    for d, h in enumerate(hs):
        with torch.cuda.device(d):
            h.reset()
    rng = np.random.default_rng(3)
    for t in range(40):
        act = random_actions(rng, N, A)
        for d, h in enumerate(hs):
            a = torch.as_tensor(act).to(f'cuda:{d}')
            with torch.cuda.device(d):
                h.step(a.data_ptr())
            torch.cuda.synchronize(d)
        for n in names:
            assert torch.equal(hs[0].tensor(n).cpu(), hs[1].tensor(n).cpu()), (t, n)
    assert hs[0].get_state().tobytes() == hs[1].get_state().tobytes()
    for h in hs:
        h.close()


def test_step_host_obs_and_async_pipeline():
    """msv_step_host_obs lands every observation tensor in host memory (one copy of the output
    arena) and equals the device tensors; the async/wait split keeps two env groups in flight."""
    import torch
    from masurvival.envs import MaSurvivalVec
    from masurvival.config import variant
    N = 300
    for name in ('2v2', 'ffa_lidar'):
        A = 4 if name == '2v2' else 8
        e1 = MaSurvivalVec(variant(name), N, seed=4)
        e2 = MaSurvivalVec(variant(name), N, seed=4)
        e1.reset(); e2.reset()
        buf, views = e2.host_obs_buffer()
        rew = torch.empty((N, A), dtype=torch.float32).pin_memory(); done = torch.empty((N,), dtype=torch.uint8).pin_memory()
        rng = np.random.default_rng(3)
        for t in range(25):
            a = random_actions(rng, N, A)
            obs, r1, d1, _ = e1.step(torch.as_tensor(a).cuda())
            if t % 2:
                e2.step_host_obs(a, buf, rew, done)
            else:
                e2.step_host_async(a, rew, done, buf); e2.step_host_wait()
            torch.cuda.synchronize()
            assert np.array_equal(r1.cpu().numpy(), rew.numpy()) and np.array_equal(d1.cpu().numpy(), done.numpy().astype(bool))
            for k, v in views.items():
                dv = e1._h.tensor(k).cpu().numpy()
                assert v.shape == dv.shape and np.array_equal(v, dv), (name, t, k)
        with pytest.raises(ValueError):
            e2.step_host(torch.zeros((N, A, 6), dtype=torch.int64), rew, done)   # wrong dtype must not reach the C ABI (numpy input is converted)
        with pytest.raises(ValueError):
            e2.step_host(np.zeros((N - 1, A, 6), dtype=np.uint8), rew, done)   # wrong size
        e1.close(); e2.close()


def test_tensor_outlives_environment():
    """ADVICE r1: closing an env while DLPack tensors are alive must not free their storage"""
    import gc
    import torch
    from masurvival.envs import MaSurvivalVec
    from masurvival.config import variant
    e = MaSurvivalVec(variant('2v2'), 128, seed=1)
    obs = e.reset()
    keep = obs['agent']; ref = keep.clone()
    rew = e._h.tensor('rewards')
    e.close()
    junk = [torch.empty(1 << 20, device='cuda').fill_(7.0) for _ in range(8)]   # would reuse freed blocks
    torch.cuda.synchronize()
    assert torch.equal(keep, ref) and float(rew.abs().sum()) == 0.0
    del keep, rew, obs, junk
    gc.collect()                                   # last export dropped -> the library frees the handle now
    e2 = MaSurvivalVec(variant('2v2'), 128, seed=1)
    assert torch.equal(e2.reset()['agent'], ref)
    e2.close()


def test_set_state_validation_and_out_of_range_actions():
    import torch
    from masurvival import _lib
    rec = make_config('2v2', auto_reset=False)
    h = _lib.Handle(rec, 8, 0, 1, 0)
    h.reset()
    s = h.get_state()
    for field, val in (('n_boxes', 9), ('n_heals', -1), ('zone_phase', 7), ('inv_n', 5)):
        bad = s.copy()
        if field == 'inv_n':
            bad[field][2][1] = val
        else:
            bad[field][2] = val
        with pytest.raises(_lib.MasurvError, match='INVALID'):
            h.set_state(bad)
    bad = s.copy(); bad['inv_n'][0][0] = 1; bad['inv_kind'][0][0][0] = 3
    with pytest.raises(_lib.MasurvError, match='INVALID'):
        h.set_state(bad)
    assert h.get_state().tobytes() == s.tobytes()          # nothing was written by the rejected calls
    # partial get/set: only the requested columns move
    part = h.get_state(first=3, count=2)
    assert part.tobytes() == s[3:5].tobytes()
    h.set_state(s[5:6], first=1)
    s2 = h.get_state()
    assert s2[1].tobytes() == s[5].tobytes() and s2[0].tobytes() == s[0].tobytes() and s2[2].tobytes() == s[2].tobytes()
    # action bytes outside MultiDiscrete([3,3,3,2,2,2]) are clamped, never index past the impulse tables
    h.close()
    h = _lib.Handle(rec, 8, 0, 1, 0); h.reset()
    a = torch.full((8, 4, 6), 255, dtype=torch.uint8, device='cuda')
    b = torch.zeros((8, 4, 6), dtype=torch.uint8, device='cuda'); b[..., :3] = 2; b[..., 3:] = 1
    h2 = _lib.Handle(rec, 8, 0, 1, 0); h2.reset()
    for _ in range(5):
        h.step(a.data_ptr()); h2.step(b.data_ptr())
    torch.cuda.synchronize()
    assert h.get_state().tobytes() == h2.get_state().tobytes()
    h.close(); h2.close()
    with pytest.raises(_lib.MasurvError, match='INVALID'):
        _lib.Handle(rec, 8, 0, 1, (1 << 32) - 4)           # global env ids must fit the 32-bit Philox counter word


def test_unwired_modules_and_episode_stats():
    """ImmunityPhase / BattleRoyale (semantics.py:652-674, 31-46) behind config keys, and the per-env
    episode_return / episode_length buffers, lock-step against the oracle"""
    import gpu_lockstep
    r = gpu_lockstep.run('1v1', 48, 160, verbose=False, modules={'immunity_phase': True, 'battle_royale': True},
                         immunity_phase={'cooldown': 7}, safe_zone={'cooldown': 6}, health={'health': 9},
                         reward_scheme={'r_alive': 0.5, 'r_dead': -0.25, 'r_kill': 3, 'r_death': -1})
    _assert_clean(r)
    assert r['episode_stats_checked'] > 40
    r = gpu_lockstep.run('2v2', 32, 120, verbose=False, modules={'immunity_phase': True, 'battle_royale': True},
                         immunity_phase={'cooldown': 0}, safe_zone={'cooldown': 6}, health={'health': 9}, gameover={'mode': 'lastalive'})
    _assert_clean(r)
    assert r['episode_stats_checked'] > 20


def test_lockstep_box2d_variants():
    """the switchable Box2D build details (clamp damping, toiCount >= maxSubSteps) are honoured identically
    by the oracle and the kernel"""
    import gpu_lockstep
    r = gpu_lockstep.run('2v2', 48, 150, verbose=False, box2d={'variant': 5})
    _assert_clean(r)
    r = gpu_lockstep.run('ffa', 16, 120, verbose=False, box2d={'variant': 7}, spawn_grid={'grid_size': 8, 'floor_size': 14},
                         safe_zone={'cooldown': 80, 'radiuses': [7, 4, 2, 1]})
    _assert_clean(r)
    assert r['toi_events'] > 0


CHECKED_CHILD = r"""
import numpy as np, torch
import parity
from masurvival import _lib
assert _lib.LIB_PATH.endswith('libmasurv_check.so')
rng = np.random.default_rng(0)
for name, n, steps, over, fwd in (('2v2', 4096, 500, {}, False),
                                  ('ffa', 1024, 300, {'spawn_grid': {'grid_size': 8, 'floor_size': 14}, 'inventory': {'slots': 1},
                                                      'safe_zone': {'cooldown': 60, 'radiuses': [7, 4, 2, 1]}}, True),
                                  ('1v1', 2048, 300, {'boxes': {'ownership': True}, 'observation': {'omniscent': False}}, False),
                                  ('ffa_lidar', 512, 100, {}, True)):
    rec = parity.make_config(name, auto_reset=True, **over)
    A = int(rec['n_agents'])
    h = _lib.Handle(rec, n, 0, 3, 0)
    h.reset()
    for t in range(steps):
        a = parity.random_actions(rng, n, A, 0.7, 0.4, 0.3)
        if fwd:
            a[..., 0] = 2                       # everybody pushes forward: pile-ups, wedges, long TOI chains
        h.step(torch.as_tensor(a).cuda().data_ptr())
    torch.cuda.synchronize()
    bad, line = h.check_failures()
    assert bad == 0, (name, bad, line)
    assert h.overflow_events() == 0, name
    st = h.flush_stats()
    assert int(st['steps']) == n * steps, (name, st)
    print(name, 'episodes', int(st['episodes']), 'steps', int(st['steps']))
    h.close()
print('CHECKED-BUILD-CLEAN')
"""


def test_checked_build():
    """compute-sanitizer is closed on the GPU pool: the bounds-checked twin of the library (make CHECK=1: every
    indexed access to the shared-memory state column and the fixed-capacity lists is range-checked) runs crowded
    roll-outs of all three capacity classes in a child process and must count zero violations and zero overflows"""
    import os
    import subprocess
    import sys
    lib = os.path.join(parity.ROOT, 'gym-ma-survival-2d_b200', 'masurvival', 'libmasurv_check.so')
    assert os.path.exists(lib), 'build it with __graft_entry__.build()'
    env = dict(os.environ, MSV_LIB=lib, PYTHONPATH=os.pathsep.join(
        [os.path.join(parity.ROOT, 'tests'), os.path.join(parity.ROOT, 'oracle'), os.path.join(parity.ROOT, 'gym-ma-survival-2d_b200')]))
    p = subprocess.run([sys.executable, '-c', CHECKED_CHILD], env=env, capture_output=True, text=True, timeout=1200)
    assert p.returncode == 0 and 'CHECKED-BUILD-CLEAN' in p.stdout, (p.stdout[-2000:], p.stderr[-4000:])
