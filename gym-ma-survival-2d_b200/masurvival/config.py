"""Config handling for the batched masurvival simulator.

Accepts the reference's nested config dict (same keys, same merge rule --
masurvival/envs/masurvival_env.py:49-54, defaults env:140-238) and flattens it
into the POD `msv_config` of include/masurv.h that crosses the C ABI."""
import copy
import math
import os

import numpy as np

from ._cstruct import parse_header

_HERE = os.path.dirname(os.path.abspath(__file__))


def _find_header():
    for cand in (os.path.join(_HERE, '..', '..', 'include', 'masurv.h'),
                 os.path.join(_HERE, '..', 'include', 'masurv.h'),
                 os.path.join(_HERE, 'masurv.h')):
        if os.path.exists(cand):
            return os.path.abspath(cand)
    raise FileNotFoundError('include/masurv.h not found next to the package')


DEFINES, STRUCTS = parse_header(_find_header())
CONFIG_DT = STRUCTS['msv_config']
STATE_DT = STRUCTS['msv_env_state']
STATS_DT = STRUCTS['msv_stats']


class CircleShape:
    """Stand-in for the reference's `sim.circle_shape(r)` config values
    (env:222-227): only the radius matters (shape_query tests body centres)."""

    def __init__(self, radius):
        self.radius = float(radius)

    def __repr__(self):
        return f'CircleShape({self.radius})'


def default_config():
    """The reference's class default (1v1, heals + boxes), env:140-238."""
    return {
        'observation': {'omniscent': True},
        'reward_scheme': {'r_alive': 1, 'r_dead': -1, 'r_kill': 0, 'r_death': 0},
        'gameover': {'mode': 'alldead'},
        'rng': {'seed': 42},
        'spawn_grid': {'grid_size': 4, 'floor_size': 20},
        'immunity_phase': {'cooldown': 300},
        'agents': {'n_agents': 2, 'agent_size': 1},
        'teams': {'twoteams': False},
        'cameras': {'fov': 0.4 * math.pi, 'depth': 10},
        'motors': {'impulse': (0.25, 0.25, 0.0125), 'drift': False},
        'health': {'health': 100},
        'melee': {'range': 2, 'damage': 20, 'cooldown': 40, 'drift': True},
        'boxes': {
            'reset_spawns': {'n_boxes': 4, 'box_size': 1},
            'ownership': False,
            'item': {'item_size': 0.5, 'offset': 0.75},
            'health': 20,
        },
        'heals': {
            'reset_spawns': {'n_items': 4, 'item_size': 0.5},
            'heal': {'healing': 50},
        },
        'inventory': {'slots': 4},
        'auto_pickup': {'shape': CircleShape(0.5)},
        'give': {'shape': CircleShape(2)},
        'death_drop': {'radius': 0.5},
        'safe_zone': {'phases': 5, 'cooldown': 100, 'damage': 1,
                      'radiuses': [10, 5, 2.5, 1], 'centers': 'random'},
        # extension (the reference's Lidars module, simulation.py:357-392, is
        # not wired into its env; off by default here as well)
        'lidars': {'n_lasers': 0, 'fov': 0.8 * math.pi, 'depth': 10},
        # modules the reference ships but never instantiates (env:322,336): opt-in.
        # ImmunityPhase takes its cooldown from 'immunity_phase' above (env:157).
        'modules': {'immunity_phase': False, 'battle_royale': False},
        # Box2D build details that cannot be pinned in this image (DESIGN.md section 4):
        # bit 0 clamp damping, bit 1 squared weld tolerance, bit 2 toiCount >= maxSubSteps
        'box2d': {'variant': 0},
    }


def merge_config(user):
    """Reference merge rule: deep copy of the defaults, then a SHALLOW
    `|=` of every user sub-dict (env:51-54)."""
    cfg = copy.deepcopy(default_config())
    continuous_melee = False
    if user is not None:
        for k, sub in user.items():
            if k not in cfg:
                cfg[k] = {}
            cfg[k].update(sub)
        # env:309-312: the melee class is chosen from the USER config
        if 'melee' not in user:
            raise KeyError('melee')
        continuous_melee = 'cooldown' not in user['melee']
    return cfg, continuous_melee


def _radius(shape):
    if hasattr(shape, 'radius'):
        return float(shape.radius)
    if isinstance(shape, dict):
        return float(shape['radius'])
    return float(shape)


OBS_LAYOUTS = ('dict', 'flat')    # msv_config.obs_layout: MSV_OBS_DICT, MSV_OBS_FLAT


def pack_config(cfg, continuous_melee=False, auto_reset=False, max_episode_steps=0, obs_layout='dict'):
    """Nested (merged) config dict -> msv_config record (numpy void).  `max_episode_steps`: the
    step limit of the vector env (0 = none), an extension the reference does not have.
    `obs_layout`: 'dict' (one tensor per observation key) or 'flat' (one [N, A, D] tensor, the keys
    as views into it; see MaSurvivalVec.flat_obs)."""
    if obs_layout not in OBS_LAYOUTS:
        raise ValueError(f"obs_layout must be 'dict' or 'flat', not {obs_layout!r}")
    rec = np.zeros((), dtype=CONFIG_DT)
    agents = cfg['agents']
    rec['n_agents'] = agents.get('n_spawns', agents.get('n_agents'))
    boxes = cfg['boxes']
    brs = boxes['reset_spawns']
    rec['n_boxes'] = brs.get('n_boxes', brs.get('n_spawns'))
    hrs = cfg['heals']['reset_spawns']
    rec['n_heals'] = hrs.get('n_items', hrs.get('n_spawns'))
    rec['teams'] = int(bool(cfg.get('teams', {}).get('twoteams', False)))
    rec['omniscient'] = int(bool(cfg['observation']['omniscent']))
    mode = cfg['gameover']['mode']
    if mode not in ('alldead', 'lastalive'):
        raise AssertionError('Invalid gameover mode')
    rec['gameover_mode'] = 0 if mode == 'alldead' else 1
    rec['grid_size'] = cfg['spawn_grid']['grid_size']
    rec['floor_size'] = cfg['spawn_grid']['floor_size']
    rec['health'] = cfg['health']['health']
    melee = cfg['melee']
    rec['melee_range'] = melee['range']
    rec['melee_damage'] = melee['damage']
    rec['melee_cooldown'] = -1 if continuous_melee else melee['cooldown']
    rec['box_ownership'] = int(bool(boxes.get('ownership', False)))
    rec['box_health'] = boxes['health']
    rec['box_size'] = brs.get('box_size', 1)
    rec['box_min_w'] = 0.1; rec['box_min_h'] = 0.1
    if 'randomized_shape' in boxes:
        rs = boxes['randomized_shape']
        rec['box_randomized'] = 1
        rec['box_avg_w'] = rs['avg_w']; rec['box_std_w'] = rs['std_w']
        rec['box_avg_h'] = rs['avg_h']; rec['box_std_h'] = rs['std_h']
        rec['box_min_w'] = rs.get('min_w', 0.1); rec['box_min_h'] = rs.get('min_h', 0.1)
    rec['box_item_size'] = boxes['item']['item_size']
    rec['box_item_offset'] = boxes['item']['offset']
    rec['heal_item_size'] = hrs['item_size']
    rec['healing'] = cfg['heals']['heal']['healing']
    rec['inv_slots'] = cfg['inventory']['slots']
    rec['pickup_radius'] = _radius(cfg['auto_pickup']['shape'])
    rec['give_radius'] = _radius(cfg['give']['shape'])
    rec['drop_radius'] = cfg['death_drop']['radius']
    sz = cfg['safe_zone']
    rec['zone_phases'] = sz['phases']
    rec['zone_cooldown'] = sz['cooldown']
    rec['zone_damage'] = sz['damage']
    radiuses = list(sz['radiuses'])
    rec['zone_n_radiuses'] = len(radiuses)
    for i, r in enumerate(radiuses):
        rec['zone_radiuses'][i] = r
    if isinstance(sz['centers'], str):
        if sz['centers'] != 'random':
            raise ValueError("safe_zone.centers must be 'random' or a list")
        rec['zone_centers_random'] = 1
    else:
        for i, c in enumerate(sz['centers']):
            rec['zone_centers'][i] = c
    rs = cfg['reward_scheme']
    rec['r_alive'] = rs.get('r_alive', 0); rec['r_dead'] = rs.get('r_dead', 0)
    rec['r_kill'] = rs.get('r_kill', 0); rec['r_death'] = rs.get('r_death', 0)
    rec['agent_size'] = agents.get('agent_size', 1)
    rec['cam_fov'] = cfg['cameras']['fov']
    rec['cam_depth'] = cfg['cameras']['depth']
    rec['motor_impulse'] = cfg['motors']['impulse']
    lid = cfg.get('lidars', {})
    rec['lidar_n'] = lid.get('n_lasers', 0)
    rec['lidar_fov'] = lid.get('fov', 0.8 * math.pi)
    rec['lidar_depth'] = lid.get('depth', 10)
    mods = cfg.get('modules', {})
    rec['immunity_cooldown'] = int(cfg.get('immunity_phase', {}).get('cooldown', 300)) if mods.get('immunity_phase') else -1
    rec['battle_royale'] = int(bool(mods.get('battle_royale', False)))
    rec['b2_variant'] = int(cfg.get('box2d', {}).get('variant', 0))
    # False/0 off, True/1 in-kernel reset, 'terminal'/2 reset + terminal observation capture
    rec['auto_reset'] = 2 if auto_reset in ('terminal', 2) else int(bool(auto_reset))
    rec['max_episode_steps'] = int(max_episode_steps)
    rec['obs_layout'] = OBS_LAYOUTS.index(obs_layout)
    validate(rec)
    return rec


def validate(rec):
    D = DEFINES
    A, B, H = int(rec['n_agents']), int(rec['n_boxes']), int(rec['n_heals'])
    if not (1 <= A <= D['MSV_MAX_AGENTS']):
        raise ValueError(f'n_agents must be in 1..{D["MSV_MAX_AGENTS"]}')
    if not (0 <= B <= D['MSV_MAX_BOXES']):
        raise ValueError(f'n_boxes must be in 0..{D["MSV_MAX_BOXES"]}')
    if not (0 <= H <= D['MSV_MAX_HEALS']):
        raise ValueError(f'n_heals must be in 0..{D["MSV_MAX_HEALS"]}')
    if A + B + H > int(rec['grid_size']) ** 2:
        # SpawnGrid.placements pops from an empty list (semantics.py:76-79)
        raise IndexError('pop from empty list: A+B+H exceeds grid_size**2')
    if int(rec['grid_size']) > 8:
        raise ValueError('grid_size must be <= 8')
    if not (1 <= int(rec['inv_slots']) <= D['MSV_MAX_SLOTS']):
        raise ValueError(f'inventory.slots must be in 1..{D["MSV_MAX_SLOTS"]}')
    if int(rec['zone_n_radiuses']) + 1 > D['MSV_MAX_ZONES']:
        raise ValueError('too many safe-zone radiuses')
    if int(rec['lidar_n']) > D['MSV_MAX_LASERS']:
        raise ValueError(f'lidars.n_lasers must be <= {D["MSV_MAX_LASERS"]}')
    if int(rec['max_episode_steps']) < 0:
        raise ValueError('max_episode_steps must be >= 0 (0: no step limit)')
    if rec['teams'] and A < 2:
        raise ValueError('teams need at least 2 agents')


# Named variants of BASELINE.json `configs` (SURVEY.md section 8d).
def variant(name):
    """User-config dicts for the benchmark variants."""
    if name == '1v1':
        return {'melee': {'cooldown': 40}}
    if name == '1v1_heal_only':
        return {'melee': {'cooldown': 40, 'damage': 0},
                'boxes': {'reset_spawns': {'n_boxes': 0, 'box_size': 1}}}
    if name == '2v2':
        return {'melee': {'cooldown': 40}, 'agents': {'n_agents': 4},
                'teams': {'twoteams': True}}
    if name in ('ffa', 'ffa_lidar'):
        u = {'melee': {'cooldown': 40}, 'agents': {'n_agents': 8},
             'spawn_grid': {'grid_size': 8},
             'boxes': {'reset_spawns': {'n_boxes': 8, 'box_size': 1},
                       'randomized_shape': {'avg_w': 1.5, 'std_w': 0.5, 'avg_h': 1.5, 'std_h': 0.5}},
             'heals': {'reset_spawns': {'n_items': 16, 'item_size': 0.5}}}
        if name == 'ffa_lidar':
            u['lidars'] = {'n_lasers': 32, 'fov': 0.8 * math.pi, 'depth': 10}
        return u
    raise KeyError(name)
