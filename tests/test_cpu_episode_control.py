"""Episode control without a device: the step-limit field of msv_config and the argument checks of
msv_create / msv_reset_envs that run before anything touches the GPU."""
import ctypes

import numpy as np
import pytest

import parity


def test_pack_config_max_episode_steps():
    from masurvival import _lib
    from masurvival.config import merge_config, pack_config
    cfg, cm = merge_config(parity.variant('2v2'))
    assert int(pack_config(cfg, cm)['max_episode_steps']) == 0
    assert int(pack_config(cfg, cm, max_episode_steps=37)['max_episode_steps']) == 37
    with pytest.raises(ValueError):
        pack_config(cfg, cm, max_episode_steps=-1)
    # the field took the place of the reserved word: same offset, same size
    assert _lib.CONFIG_DT.itemsize == _lib.load().msv_sizeof_config()
    assert _lib.CONFIG_DT.fields['max_episode_steps'][1] == _lib.CONFIG_DT.fields['b2_variant'][1] + 4


def test_create_refuses_negative_limit_before_the_device():
    from masurvival import _lib
    L = _lib.load()
    rec = np.array(parity.make_config('2v2'), dtype=_lib.CONFIG_DT).reshape(1)
    rec['max_episode_steps'] = -5
    h = ctypes.c_void_p()
    assert L.msv_create(rec.ctypes.data, 8, 0, 1, 0, ctypes.byref(h)) == -1     # MSV_ERR_INVALID, not NO_DEVICE
    assert not h.value


def test_reset_envs_null_arguments():
    from masurvival import _lib
    assert _lib.load().msv_reset_envs(None, None, None) == -1
