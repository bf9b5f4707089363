"""The lidar against a float64 restatement of Lidars._update (simulation.py:377-392) that shares no code
with b2lite: exact ray/circle and ray/slab intersections with the agents, the item and heal sensors, the
boxes and the four ThickRoomWalls.  The oracle (b2lite's b2l_raycast) must agree with it on every
well-conditioned ray, on crafted scenes around the fan edges and on roll-out states.  The golden
fixtures and the GPU lidar are both compared with the oracle, so this pins the ray geometry itself."""
import math

import numpy as np
import pytest

import obs_cases as oc
import parity

# (A, L, fov, depth): every fan width on both sides of the kernel's non-convex cull threshold
# (A, L, fov, depth, least well-conditioned share of the rays): every fan width on both sides of the kernel's
# non-convex cull threshold.  The crafted scenes put bodies on the fan edges, at the segment's end +- eps and on a
# tangent on purpose, so the narrow fans (where those rays are most of the fan) keep only about three quarters
# of their rays; the floors sit a little under what each scene set measures, so a change that made the filter
# drop more rays fails here instead of quietly shrinking the comparison.
CONFIGS = [(1, 1, 0.1, 10.0, 0.72), (2, 9, 0.8 * math.pi, 2.0, 0.72), (3, 31, 2.95, 30.0, 0.95), (4, 32, math.pi, 10.0, 0.97),
           (5, 2, 1.5 * math.pi, 0.4, 0.96), (8, 32, 2 * math.pi, 10.0, 0.96), (4, 9, 3.2, 10.0, 0.83)]


def _compare(rec, states, seen):
    import pyoracle as po
    bad, n_good, n_all = [], 0, 0
    o = po.OracleEnv(rec, seed=3, env_id=0)
    o.reset()
    depth = float(rec['lidar_depth'])
    for tag, s in states:
        o.set_state(s)
        out = o.observe()
        f, h, good = oc.lidar_reference(rec, s)
        alive = s['alive'][:int(rec['n_agents'])] != 0
        n_all += int(good[alive].size); n_good += int(good[alive].sum())
        for i, r in zip(*np.nonzero(good)):
            seen.add(int(h[i, r]) >> 8)
            if out['lidar_hit'][i, r] != h[i, r] or abs(float(out['lidar_frac'][i, r]) - f[i, r]) * depth > 1e-4:
                bad.append((tag, int(i), int(r), int(out['lidar_hit'][i, r]), int(h[i, r]), float(out['lidar_frac'][i, r]), f[i, r]))
        dead = ~alive
        assert np.all(out['lidar_frac'][dead] == 1.0) and np.all(out['lidar_hit'][dead] == 0), tag
    o.close()
    return bad, n_good, n_all


@pytest.mark.parametrize('A,L,fov,depth,least', CONFIGS)
def test_reference_matches_oracle_on_crafted_scenes(A, L, fov, depth, least):
    import pyoracle as po
    rec = oc.lidar_config(A, L, fov, depth)
    o = po.OracleEnv(rec, seed=5, env_id=1)
    o.reset()
    base = o.get_state(); o.close()
    rng = np.random.default_rng(A * 100 + L)
    states = oc.lidar_states(rec, base, rng)
    seen = set()
    bad, n_good, n_all = _compare(rec, states, seen)
    assert not bad, bad[:8]
    assert n_good >= least * n_all, 'well-conditioned %d of %d rays (%.1f %% excluded)' % (n_good, n_all, 100 - 100 * n_good / n_all)
    assert oc.KIND_WALL in seen or depth < 1


ROLLOUTS = {
    'ffa_lidar': lambda: parity.make_config('ffa_lidar'),
    'a7_lidar': lambda: oc.matrix_config(dict((m[0], m[2]) for m in oc.MATRIX)['a7_lidar']),
    'ffa_fan3.2_depth30': lambda: parity.make_config('ffa', lidars={'n_lasers': 31, 'fov': 3.2, 'depth': 30}),
    '1v1_one_ray': lambda: parity.make_config('1v1', lidars={'n_lasers': 1, 'fov': 0.1, 'depth': 10}),
}


@pytest.mark.parametrize('name', sorted(ROLLOUTS))
def test_reference_matches_oracle_on_rollouts(name):
    import pyoracle as po
    rec = ROLLOUTS[name]()
    A = int(rec['n_agents'])
    rng = np.random.default_rng(7)
    states, seen = [], set()
    for env in range(3):
        o = po.OracleEnv(rec, seed=11, env_id=env)
        o.reset()
        for t in range(200):
            a = parity.random_actions(rng, 1, A, 0.6, 0.5, 0.3)[0]
            a[:, 0] = rng.integers(1, 3, size=A)              # mostly forward: agents reach walls and each other
            if o.step(a)['done']:
                o.reset()
            if t % 10 == 9:
                states.append(('env%d_t%d' % (env, t), o.get_state()))
        o.close()
    bad, n_good, n_all = _compare(rec, states, seen)
    assert not bad, bad[:8]
    assert n_good >= 0.95 * n_all, 'well-conditioned %d of %d rays (%.1f %% excluded)' % (n_good, n_all, 100 - 100 * n_good / n_all)
    assert oc.KIND_WALL in seen
