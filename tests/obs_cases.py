"""Shared builders for the config-matrix and lidar tests: the matrix of agent counts and capacity
classes, crafted msv_env_state records (dead agents, inventories, list lengths at 0 and at their
maximum, last zone phase, bodies placed on and around the lidar fan), and a float64 restatement of
the reference's Lidars._update (simulation.py:377-392) that shares no code with b2lite."""
import math

import numpy as np

import parity
from parity import make_config, scramble_state

# ---------------------------------------------------------------- the matrix
# Short zone phases and little health: every entry sees deaths, death drops and in-kernel resets.
FAST = {'safe_zone': {'cooldown': 8}, 'health': {'health': 12}}
TEAMS = {'teams': {'twoteams': True}}
PARTIAL = {'observation': {'omniscent': False}}


def _heals(n):
    return {'heals': {'reset_spawns': {'n_items': n, 'item_size': 0.5}}}


def _boxes(n):
    return {'boxes': {'reset_spawns': {'n_boxes': n, 'box_size': 1}}}


def _agents(n):
    return {'agents': {'n_agents': n, 'agent_size': 1}}


def _merge(*parts):
    out = {}
    for p in parts:
        for k, v in p.items():
            out.setdefault(k, {}).update(v)
    return out


# (id, variant, overrides, capacity class).  Class 0/1/2 runs G = 2/4/8 lanes per environment.
MATRIX = [
    ('a1_default', '1v1', _merge(_agents(1)), 0),
    ('a1_heals8', '1v1', _merge(_agents(1), _heals(8)), 2),
    ('a2_heals6', '1v1', _merge(_agents(2), _heals(6)), 2),
    ('a3_teams', '1v1', _merge(_agents(3), TEAMS), 1),
    ('a3_partial', '1v1', _merge(_agents(3), PARTIAL), 1),
    ('a4_boxes6_teams', '1v1', _merge(_agents(4), _boxes(6), TEAMS), 2),
    ('a5_teams', '1v1', _merge(_agents(5), TEAMS), 2),
    ('a6_partial', '1v1', _merge(_agents(6), PARTIAL), 2),
    ('a7_lidar', '1v1', _merge(_agents(7), {'lidars': {'n_lasers': 9, 'fov': 0.8 * math.pi, 'depth': 10}}), 2),
]
LANES = {0: 2, 1: 4, 2: 8}

# the observation tensors the library stores (msv_tensor_info names), lidar aside
OBS_KEYS = ('agent', 'others', 'others_mask', 'zone', 'heals', 'heals_mask', 'heal_slot', 'heal_slot_mask',
            'boxes', 'boxes_mask', 'box_items', 'box_items_mask', 'box_slot', 'box_slot_mask')


def terminal_snapshot(h):
    """copies of a terminal-mode handle's terminal_<key> observation tensors (terminal_lidar_* left out:
    the terminal k_lidar rewrites every row on every step)"""
    names = ['terminal_' + k for k in OBS_KEYS]
    return {n: h.tensor(n).clone() for n in names if h.has_tensor(n)}


def assert_unfinished_rows_kept(h, snap, finished, where=None):
    """the rows of environments that did not finish on the step are the bytes they held before it"""
    import torch
    keep = torch.as_tensor(finished).to('cuda') == 0
    for n, before in snap.items():
        assert torch.equal(h.tensor(n)[keep].view(torch.int32), before[keep].view(torch.int32)), (where, n)


def matrix_config(over, auto_reset=False, fast=True):
    return make_config('1v1', auto_reset=auto_reset, **_merge(FAST if fast else {}, over))


def plan_class(rec, n_envs=37):
    """capacity class from msv_plan_tile (host logic, no device needed)"""
    import ctypes
    from masurvival import _lib
    L = _lib.load()
    buf = np.array(rec, dtype=_lib.CONFIG_DT).reshape(1)
    out = (ctypes.c_int32 * 4)()
    _lib.check(L.msv_plan_tile(buf.ctypes.data, n_envs, 148, 227 * 1024, out))
    return int(out[3])


# ------------------------------------------------------------ crafted states
def kill(s, i):
    """agent i dead, in the form the oracle leaves a dead agent (everything zero but the cause)"""
    for f in ('alive', 'health', 'cooldown', 'x', 'y', 'angle', 'vx', 'vy', 'omega', 'sleep_time', 'awake', 'inv_n'):
        s[f][i] = 0
    s['fat'][i] = 0
    s['inv_kind'][i] = 0; s['inv_owner'][i] = 0
    s['inv_shape'][i] = np.zeros_like(s['inv_shape'][i])
    s['pair_aa'] = np.zeros_like(s['pair_aa']); s['pair_ab'] = np.zeros_like(s['pair_ab']); s['pair_aw'] = np.zeros_like(s['pair_aw'])


def fit_fat(s, rec, i):
    r = np.float32(rec['agent_size'] / 2); ext = np.float32(0.1)
    x, y = s['x'][i], s['y'][i]
    s['fat'][i] = [(x - r) - ext, (y - r) - ext, (x + r) + ext, (y + r) + ext]


def set_items(s, rec, n, rng):
    """n box items on the floor at random places (items come from broken boxes: newer bodies)"""
    s['n_items'] = n
    for k in range(s['item_x'].shape[0]):
        if k < n:
            s['item_x'][k], s['item_y'][k] = np.float32(rng.uniform(-8, 8)), np.float32(rng.uniform(-8, 8))
            s['item_shape'][k]['hx'] = np.float32(rng.uniform(0.3, 0.8)); s['item_shape'][k]['hy'] = np.float32(rng.uniform(0.3, 0.8))
            s['item_shape'][k]['rehulled'] = 1
            s['item_owner'][k] = -1
            s['item_seq'][k] = int(s['body_seq']); s['body_seq'] += 1
        else:
            s['item_x'][k] = s['item_y'][k] = 0; s['item_owner'][k] = 0; s['item_seq'][k] = 0
            s['item_shape'][k] = np.zeros((), dtype=s['item_shape'].dtype)


def truncate_lists(s, nb, nh):
    s['n_boxes'] = nb; s['n_heals'] = nh
    for k in range(nb, s['box_x'].shape[0]):
        for f in ('box_x', 'box_y', 'box_health', 'box_has_health', 'box_cause', 'box_owner', 'box_seq'):
            s[f][k] = 0
        s['box_shape'][k] = np.zeros((), dtype=s['box_shape'].dtype)
    for k in range(nh, s['heal_x'].shape[0]):
        s['heal_x'][k] = 0; s['heal_y'][k] = 0; s['heal_seq'][k] = 0
    s['pair_ab'] = np.zeros_like(s['pair_ab'])


def items_in_view(rec, base, rng):
    """`base` with box items on the floor 2-4 m in front of the agents (inside their camera cone), and
    as many boxes removed as there are items, so that boxes + items never exceed what a reset created"""
    A, B = int(rec['n_agents']), int(rec['n_boxes'])
    n = min(2, B)
    s = base.copy()
    truncate_lists(s, B - n, int(s['n_heals']))
    set_items(s, rec, n, rng)
    alive = [i for i in range(A) if s['alive'][i]]
    for k in range(n):
        i = alive[k % len(alive)]
        a = float(s['angle'][i]) + rng.uniform(-0.3, 0.3)
        d = rng.uniform(2.0, 4.0)
        s['item_x'][k] = np.float32(np.clip(s['x'][i] + d * math.cos(a), -9.3, 9.3))
        s['item_y'][k] = np.float32(np.clip(s['y'][i] + d * math.sin(a), -9.3, 9.3))
    return s


def observation_states(rec, base, rng):
    """(tag, state) pairs for the observation-of-injected-state tests, all derived from the
    freshly reset state `base` of an environment of `rec`"""
    A, B, H = int(rec['n_agents']), int(rec['n_boxes']), int(rec['n_heals'])
    slots = int(rec['inv_slots'])
    out = [('reset', base.copy())]
    for q in range(2):
        out.append(('scrambled%d' % q, scramble_state(base, rec, rng)))
    s = scramble_state(base, rec, rng)                  # dead agents: the first and the last (the rank remap, dead rows)
    kill(s, 0)
    if A > 1:
        kill(s, A - 1)
    out.append(('dead_first_last', s))
    s = scramble_state(base, rec, rng)                  # a heal / a box on top of an inventory
    for i in range(A):
        n = slots
        s['inv_n'][i] = n
        for k in range(n):
            top = k == n - 1
            kind = (1 if i % 2 == 0 or B == 0 else 2) if top else (2 if (k + i) % 2 and B > 0 else 1)
            s['inv_kind'][i][k] = kind
            if kind == 2:
                s['inv_shape'][i][k]['hx'] = np.float32(0.3 + 0.1 * k); s['inv_shape'][i][k]['hy'] = np.float32(0.6)
                s['inv_shape'][i][k]['rehulled'] = 1
                s['inv_owner'][i][k] = (100 + i % 2) if rec['teams'] else i
            else:
                s['inv_shape'][i][k] = np.zeros((), dtype=s['inv_shape'].dtype); s['inv_owner'][i][k] = -1
    out.append(('carried_on_top', s))
    s = base.copy()                                     # every list empty
    truncate_lists(s, 0, 0); set_items(s, rec, 0, rng)
    out.append(('lists_empty', s))
    s = base.copy()                                     # every list at its reachable maximum
    set_items(s, rec, B, rng)
    out.append(('lists_full', s))
    s = scramble_state(base, rec, rng)                  # last zone phase: the next-zone columns are zero
    s['zone_phase'] = int(rec['zone_phases']) - 1
    s['zone_cur_r'] = np.float32(0.5); s['zone_endgame'] = 1
    out.append(('zone_last_phase', s))
    return out


# -------------------------------------------------------- lidar reference
KIND_AGENT, KIND_BOX, KIND_ITEM, KIND_HEAL, KIND_WALL = 1, 2, 3, 4, 5
TOL = 1e-4


def ray_angles(rec):
    L, fov = int(rec['lidar_n']), float(rec['lidar_fov'])
    return [r * (fov / (L - 1)) - fov / 2. if L > 1 else 0.0 for r in range(L)]


def world_bodies(rec, s):
    """every body a lidar ray can hit, as (kind, index, shape); shape is ('c', cx, cy, r) or
    ('b', cx, cy, hx, hy) (axis-aligned), in float64 from the state's float32 values"""
    A = int(rec['n_agents'])
    f = lambda v: float(np.float32(v))
    out = []
    for k in range(int(s['n_boxes'])):
        out.append((KIND_BOX, k, ('b', f(s['box_x'][k]), f(s['box_y'][k]), f(s['box_shape'][k]['hx']), f(s['box_shape'][k]['hy']))))
    for k in range(int(s['n_items'])):
        out.append((KIND_ITEM, k, ('c', f(s['item_x'][k]), f(s['item_y'][k]), rec['box_item_size'] / 2)))
    for k in range(int(s['n_heals'])):
        out.append((KIND_HEAL, k, ('c', f(s['heal_x'][k]), f(s['heal_y'][k]), rec['heal_item_size'] / 2)))
    o, t = rec['floor_size'] / 2, rec['floor_size'] / 100 / 2     # ThickRoomWalls: floor/100 thick, centred at +-floor/2
    for k, (cx, cy, hx, hy) in enumerate([(-o, 0, t, o), (0, o, o, t), (o, 0, t, o), (0, -o, o, t)]):   # W, N, E, S
        out.append((KIND_WALL, k, ('b', cx, cy, hx, hy)))
    for i in range(A):
        if s['alive'][i]:
            out.append((KIND_AGENT, i, ('c', f(s['x'][i]), f(s['y'][i]), rec['agent_size'] / 2)))
    return out


def _ray_circle(px, py, dx, dy, cx, cy, r):
    """entry fraction of p + t d, t in [0, 1], into the circle; None if the origin is inside or no entry.
    Also returns whether the ray's line is near tangency, and the origin's distance to the circle."""
    sx, sy = px - cx, py - cy
    dd = dx * dx + dy * dy
    b = sx * dx + sy * dy
    c = sx * sx + sy * sy - r * r
    perp = abs(sx * dy - sy * dx) / math.sqrt(dd)
    # Box2D's float32 formula loses |s|^2 * 2^-24 to cancellation in sigma = c^2 - rr * b, and divides it by
    # the half chord sqrt(r^2 - perp^2): a ray is near tangency when that error reaches the tolerance
    q = abs(r * r - perp * perp)
    near = abs(perp - r) < TOL or 2 * 2.0 ** -24 * (sx * sx + sy * sy) >= TOL * math.sqrt(q)
    origin_gap = abs(math.sqrt(sx * sx + sy * sy) - r)
    if c < 0:
        return None, near, origin_gap
    disc = b * b - dd * c
    if disc < 0:
        return None, near, origin_gap
    t = (-b - math.sqrt(disc)) / dd
    return (t if 0 <= t <= 1 else None), near, origin_gap


def _ray_box(px, py, dx, dy, cx, cy, hx, hy):
    """slab entry fraction into the axis-aligned box; None if the origin is inside or no entry.
    Also returns the distance from the entry point to the nearest corner, and from the origin to the boundary."""
    lo, hi = 0.0, 1.0
    entered = False
    for p, d, c, h in ((px, dx, cx, hx), (py, dy, cy, hy)):
        a, b = c - h - p, c + h - p
        if d == 0:
            if a > 0 or b < 0:
                return None, math.inf, math.inf
            continue
        t0, t1 = a / d, b / d
        if t0 > t1:
            t0, t1 = t1, t0
        if t0 > lo:
            lo, entered = t0, True
        hi = min(hi, t1)
        if lo > hi:
            return None, math.inf, math.inf
    inside_x, inside_y = abs(px - cx) - hx, abs(py - cy) - hy
    origin_gap = abs(max(inside_x, inside_y)) if max(inside_x, inside_y) < 0 else math.hypot(max(inside_x, 0), max(inside_y, 0))
    if not entered:
        return None, math.inf, origin_gap
    ex, ey = px + lo * dx, py + lo * dy
    corner = min(math.hypot(ex - (cx + sx * hx), ey - (cy + sy * hy)) for sx in (-1, 1) for sy in (-1, 1))
    return lo, corner, origin_gap


def _segment_gap(px, py, dx, dy, shape):
    """distance from the segment's end point to the shape's boundary (a body at depth +- eps)"""
    ex, ey = px + dx, py + dy
    if shape[0] == 'c':
        return abs(math.hypot(ex - shape[1], ey - shape[2]) - shape[3])
    _, cx, cy, hx, hy = shape
    qx, qy = abs(ex - cx) - hx, abs(ey - cy) - hy
    return math.hypot(max(qx, 0), max(qy, 0)) if max(qx, qy) > 0 else -max(qx, qy)


def lidar_reference(rec, s):
    """float64 Lidars._update for one environment: (frac[A, L], hit[A, L], well_conditioned[A, L])"""
    A, L, depth = int(rec['n_agents']), int(rec['lidar_n']), float(rec['lidar_depth'])
    frac = np.ones((A, L)); hit = np.zeros((A, L), dtype=np.int32); good = np.ones((A, L), dtype=bool)
    bodies = world_bodies(rec, s)
    angs = ray_angles(rec)
    for i in range(A):
        if not s['alive'][i]:
            continue                                           # dead agents: fraction 1, no hit
        px, py = float(np.float32(s['x'][i])), float(np.float32(s['y'][i]))
        for r in range(L):
            th = float(np.float32(angs[r] + float(s['angle'][i])))   # Box2D takes the angle as float32
            dx, dy = depth * math.cos(th), depth * math.sin(th)
            hits, marginal = [], False
            for kind, idx, shp in bodies:
                if kind == KIND_AGENT and idx == i:
                    continue                                   # the origin is inside: never hit
                if shp[0] == 'c':
                    t, near, og = _ray_circle(px, py, dx, dy, shp[1], shp[2], shp[3])
                else:
                    t, m, og = _ray_box(px, py, dx, dy, *shp[1:])
                    near = t is not None and m < TOL
                if og < TOL or abs(_segment_gap(px, py, dx, dy, shp)) < TOL:
                    marginal = True
                if t is not None:
                    hits.append((t, kind, idx, near))
                elif near and shp[0] == 'c':
                    # a near-tangent miss counts only if the tangent point lies on the segment
                    sx, sy = shp[1] - px, shp[2] - py
                    along = (sx * dx + sy * dy) / (depth * depth)
                    marginal |= -TOL <= along <= 1 + TOL
            hits.sort(key=lambda h: h[0])
            if hits:
                t, kind, idx, near = hits[0]
                frac[i, r] = t; hit[i, r] = (kind << 8) | idx
                if near or (len(hits) > 1 and hits[1][0] - t <= TOL):
                    marginal = True
            good[i, r] = not marginal
    return frac, hit, good


# ------------------------------------------------------ crafted lidar scenes
def _place(s, kind, idx, x, y):
    x, y = np.float32(np.clip(x, -9.3, 9.3)), np.float32(np.clip(y, -9.3, 9.3))
    if kind == 'heal':
        s['heal_x'][idx], s['heal_y'][idx] = x, y
    elif kind == 'box':
        s['box_x'][idx], s['box_y'][idx] = x, y
    elif kind == 'item':
        s['item_x'][idx], s['item_y'][idx] = x, y
    else:
        s['x'][idx], s['y'][idx] = x, y


def _movable(s, rec, observer):
    A = int(rec['n_agents'])
    out = [('heal', k) for k in range(int(s['n_heals']))] + [('item', k) for k in range(int(s['n_items']))]
    out += [('box', k) for k in range(int(s['n_boxes']))] + [('agent', i) for i in range(A) if i != observer and s['alive'][i]]
    return out


def _finish(s, rec):
    for i in range(int(rec['n_agents'])):
        if s['alive'][i]:
            fit_fat(s, rec, i)
    s['pair_aa'] = np.zeros_like(s['pair_aa']); s['pair_ab'] = np.zeros_like(s['pair_ab']); s['pair_aw'] = np.zeros_like(s['pair_aw'])
    return s


HEADINGS = [0.0, math.pi, -math.pi, math.pi / 2, -math.pi / 2, 1234.5678, -98765.4321, 1e5, -1e5]


def lidar_states(rec, base, rng):
    """(tag, state) scenes around agent 0 (the observer) of a reset state `base`: bodies on a fan edge
    and at +-1e-4, 1e-3, 1e-2 rad from it, at depth +- bound +- eps, a tangent ray, two bodies at the same
    distance, the observer inside a box, pressed into a wall; each at several headings"""
    A = int(rec['n_agents'])
    fov, depth = float(rec['lidar_fov']), float(rec['lidar_depth'])
    ra, hr = rec['agent_size'] / 2, rec['heal_item_size'] / 2
    base = base.copy()
    set_items(base, rec, min(2, int(rec['n_boxes'])), rng)
    out = []
    for hq, head in enumerate(HEADINGS):
        s0 = base.copy()
        ox, oy = rng.uniform(-2, 2), rng.uniform(-2, 2)
        s0['x'][0], s0['y'][0], s0['angle'][0] = np.float32(ox), np.float32(oy), np.float32(head)
        h = float(np.float32(head))
        mov = _movable(s0, rec, 0)
        dist = lambda k: min(1.2 + 0.9 * k, max(1.2, depth - 0.5))
        # fan edges, exactly and at +-1e-4, 1e-3, 1e-2 rad
        for delta in (0.0, 1e-4, -1e-4, 1e-3, -1e-3, 1e-2, -1e-2):
            s = s0.copy()
            for k, (kind, idx) in enumerate(mov):
                edge = (fov / 2 if k % 2 == 0 else -fov / 2) if int(rec['lidar_n']) > 1 else 0.0
                a = h + edge + delta
                _place(s, kind, idx, ox + dist(k) * math.cos(a), oy + dist(k) * math.sin(a))
            out.append(('edge%+g_h%d' % (delta, hq), _finish(s, rec)))
        # circles whose rim just reaches the outer fan edge (centre 0.9 radius outside it), far out
        s = s0.copy()
        for k, (kind, idx) in enumerate(mov):
            rad = {'heal': hr, 'item': rec['box_item_size'] / 2, 'agent': ra}.get(kind)
            if rad is None:
                continue
            side = 1 if k % 2 == 0 else -1
            a = h + side * (fov / 2 if int(rec['lidar_n']) > 1 else 0.0)
            d = max(0.3, depth - rad - 0.1 * k)
            n = side * 0.9 * rad
            _place(s, kind, idx, ox + d * math.cos(a) - n * math.sin(a), oy + d * math.sin(a) + n * math.cos(a))
        out.append(('rim_h%d' % hq, _finish(s, rec)))
        if hq % 3:
            continue
        # bodies whose near side (centre at depth + bound) or far side (centre at depth - bound) is at the
        # segment's end +- eps, straight ahead and along the other rays.  The observer stands back from the
        # room's centre so that the straight-ahead reach stays inside the walls; depth 30 is longer than the
        # room's diagonal, so there _place clamps the bodies against the walls and the scene tests the walls.
        angs = ray_angles(rec)
        back = min((depth + 0.6) / 2, 8.5)
        bx, by = -back * math.cos(h), -back * math.sin(h)
        for side in (1, -1):
            for eps in (-1e-3, -1e-4, 1e-4, 1e-3):
                s = s0.copy()
                s['x'][0], s['y'][0] = np.float32(bx), np.float32(by)
                for k, (kind, idx) in enumerate(mov):
                    a = h + angs[k % len(angs)]
                    if kind == 'box':
                        c, sn = abs(math.cos(a)), abs(math.sin(a))
                        hx, hy = float(s['box_shape'][idx]['hx']), float(s['box_shape'][idx]['hy'])
                        bound = min(hx / c if c > 1e-9 else math.inf, hy / sn if sn > 1e-9 else math.inf)
                    else:
                        bound = {'heal': hr, 'item': rec['box_item_size'] / 2, 'agent': ra}[kind]
                    d = depth + side * bound + eps
                    if d <= ra + bound + 0.01:
                        continue                                 # would overlap the observer
                    _place(s, kind, idx, bx + d * math.cos(a), by + d * math.sin(a))
                out.append(('depth%s%+g_h%d' % ('+' if side > 0 else '-', eps, hq), _finish(s, rec)))
        # a ray tangent to a circle, and two identical circles at the same place (the tie rule)
        s = s0.copy()
        circles = [m for m in mov if m[0] in ('heal', 'item', 'agent')]
        if circles:
            kind, idx = circles[0]
            rad = {'heal': hr, 'item': rec['box_item_size'] / 2, 'agent': ra}[kind]
            d = min(3.0, depth * 0.6)
            _place(s, kind, idx, ox + d * math.cos(h) - rad * math.sin(h), oy + d * math.sin(h) + rad * math.cos(h))
        out.append(('tangent_h%d' % hq, _finish(s, rec)))
        heals = [m for m in mov if m[0] == 'heal']
        if len(heals) >= 2:
            s = s0.copy()
            d = min(2.0, depth * 0.5)
            ties = heals[:2] + [m for m in mov if m[0] == 'item'][:1]     # an item is newer than every heal
            for kind, idx in ties:
                _place(s, kind, idx, ox + d * math.cos(h), oy + d * math.sin(h))
            out.append(('tie_h%d' % hq, _finish(s, rec)))
        # the observer inside a box, and pressed into each wall
        if int(s0['n_boxes']) > 0:
            s = s0.copy()
            s['x'][0], s['y'][0] = s['box_x'][0], s['box_y'][0]
            out.append(('inside_box_h%d' % hq, _finish(s, rec)))
        o, t = rec['floor_size'] / 2, rec['floor_size'] / 200
        for w, (x, y) in enumerate([(-o + t + ra - 0.02, oy), (ox, o - t - ra + 0.02), (o - t - ra + 0.02, oy), (ox, -o + t + ra - 0.02)]):
            s = s0.copy()
            s['x'][0], s['y'][0] = np.float32(x), np.float32(y)
            out.append(('wall%d_h%d' % (w, hq), _finish(s, rec)))
    return out


def lidar_config(A, L, fov, depth):
    return make_config('1v1', auto_reset=False, **_merge(_agents(A), {'lidars': {'n_lasers': L, 'fov': fov, 'depth': depth}}))
