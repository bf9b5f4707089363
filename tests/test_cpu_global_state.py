"""msv_global_state_dim (host logic, no device): the width of the global-state row for the shipped variants, for
every entry of the config matrix, and its refusal of configs out of capacity."""
import numpy as np
import pytest

import obs_cases as oc
import parity


def _formula(rec):
    A, B, H = int(rec['n_agents']), int(rec['n_boxes']), int(rec['n_heals'])
    S = 8 + (1 if rec['teams'] else 0)
    return A * (S + 1) + 6 + (3 * H + 2 * A if H > 0 else 0) + (23 * B + 9 * A if B > 0 else 0) + 1


def _dim(rec):
    from masurvival import _lib
    buf = np.array(rec, dtype=_lib.CONFIG_DT).reshape(1)
    return _lib.load().msv_global_state_dim(buf.ctypes.data)


@pytest.mark.parametrize('name,ds', [('1v1', 151), ('2v2', 195), ('1v1_heal_only', 41), ('ffa', 399), ('ffa_lidar', 399)])
def test_global_state_dim_of_the_variants(name, ds):
    from masurvival import _lib
    rec = parity.make_config(name)
    assert _dim(rec) == ds == _formula(rec)
    assert _lib.global_state_dim(rec) == ds


@pytest.mark.parametrize('cid,over', [(m[0], m[2]) for m in oc.MATRIX], ids=[m[0] for m in oc.MATRIX])
def test_global_state_dim_matches_the_formula(cid, over):
    from masurvival import _lib
    rec = oc.matrix_config(over)
    assert _dim(rec) == _formula(rec) == _lib.global_state_dim(rec)


def test_global_state_dim_largest_row():
    rec = parity.make_config('1v1', agents={'n_agents': 8, 'agent_size': 1}, teams={'twoteams': True},
                             boxes={'reset_spawns': {'n_boxes': 8, 'box_size': 1}},
                             heals={'reset_spawns': {'n_items': 16, 'item_size': 0.5}}, spawn_grid={'grid_size': 8})
    assert _dim(rec) == _formula(rec) == 407


def test_global_state_dim_refuses_bad_configs():
    from masurvival import _lib
    L = _lib.load()
    assert L.msv_global_state_dim(None) == -1
    for field, value in (('n_agents', 9), ('n_agents', 0), ('n_boxes', 9), ('n_heals', 17), ('n_boxes', -1)):
        rec = parity.make_config('2v2')
        rec[field] = value
        assert _dim(rec) == -1, field
        with pytest.raises(_lib.MasurvError):
            _lib.global_state_dim(rec)
