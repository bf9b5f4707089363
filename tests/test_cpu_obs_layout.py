"""The observation layout option (msv_config.obs_layout) on the host: the config field and its refusals,
the struct layout and ABI version the Python side checks, and the width D of a flat row."""
import ctypes

import numpy as np
import pytest

import obs_cases as oc
import parity
from masurvival import _lib
from masurvival.config import CONFIG_DT, DEFINES, merge_config, pack_config, variant


def test_obs_layout_field():
    cfg, cm = merge_config(variant('2v2'))
    assert pack_config(cfg, cm)['obs_layout'] == DEFINES['MSV_OBS_DICT'] == 0
    assert pack_config(cfg, cm, obs_layout='dict')['obs_layout'] == 0
    assert pack_config(cfg, cm, obs_layout='flat')['obs_layout'] == DEFINES['MSV_OBS_FLAT'] == 1
    assert pack_config(cfg, cm, obs_layout='flat')['reserved1'] == 0
    for bad in ('Flat', 'dicts', 1, None):
        with pytest.raises(ValueError):
            pack_config(cfg, cm, obs_layout=bad)
    from masurvival.envs import MaSurvivalVec
    with pytest.raises(ValueError):                   # refused before a handle (or a device) is needed
        MaSurvivalVec(variant('2v2'), 4, obs_layout='nested')


def test_config_struct_and_abi_version():
    L = _lib.load()
    assert CONFIG_DT.itemsize == L.msv_sizeof_config()
    assert L.msv_abi_version() == DEFINES['MSV_ABI_VERSION'] == 3
    names = CONFIG_DT.names
    assert names[-3:] == ('max_episode_steps', 'obs_layout', 'reserved1')


def test_create_refuses_bad_layout_before_touching_the_device():
    L = _lib.load()
    good = np.array(parity.make_config('2v2'), dtype=CONFIG_DT).reshape(1)
    h = ctypes.c_void_p()
    for field, val in (('obs_layout', 2), ('obs_layout', -1), ('reserved1', 1), ('reserved1', -7)):
        bad = good.copy(); bad[0][field] = val
        assert L.msv_create(bad.ctypes.data, 4, 0, 0, 0, ctypes.byref(h)) == -1, (field, val)   # MSV_ERR_INVALID


def _row_width(user):
    from masurvival.envs import MaSurvivalVec

    class Shapes(MaSurvivalVec):
        def __init__(self, user):
            self.config, cm = merge_config(user)
            self._rec = pack_config(self.config, cm, obs_layout='flat')
    return sum(int(np.prod(s[1:])) for k, s in Shapes(user).obs_shapes().items() if k != 'lidar_hit')


def test_flat_row_width():
    """D: every key of observation_space once per agent (the keys stored once per env repeated)"""
    assert {v: _row_width(variant(v)) for v in ('2v2', '1v1_heal_only', 'ffa', 'ffa_lidar')} == \
        {'2v2': 160, '1v1_heal_only': 37, 'ffa': 320, 'ffa_lidar': 352}
    # the largest capacity: A = 8, S = 9 (teams), B = 8, H = 16, L = 32
    big = oc._merge(variant('ffa_lidar'), oc.TEAMS)
    assert _row_width(big) == 360
