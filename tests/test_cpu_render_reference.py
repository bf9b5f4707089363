"""Known answers of the render reference (tests/render_reference.py), which the GPU test holds msv_render to
bit for bit, and a round trip of demo.py's PNG writer.  No device needed."""
import os
import sys

import numpy as np

import obs_cases as oc
import render_reference as rr
from parity import make_config
from masurvival import _lib
from masurvival.config import STATE_DT

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32


def _empty_state(rec):
    """no bodies, no agents, a zone wider than the picture, last zone phase (no next ring)"""
    s = np.zeros(1, dtype=STATE_DT)[0]
    s['zone_phase'] = int(rec['zone_phases']) - 1
    s['zone_cur_r'] = f32(100)
    return s


def _agent(s, i, x, y, angle=np.pi / 2):
    s['alive'][i] = 1
    s['x'][i], s['y'][i], s['angle'][i] = f32(x), f32(y), f32(angle)


def _col(rec, W, x):
    """column whose pixel centre is nearest to x (on a square image)"""
    _, xs, _ = rr.pixel_centres(rec, W, W)
    return int(np.argmin(np.abs(xs - f32(x))))


REC = make_config('1v1')
N_PX = 101                                              # odd: pixel (50, 50) is centred on the origin


def _draw(s, rec=REC, n=N_PX, frac=None):
    return rr.render_indices(rec, s, n, n, frac)


def test_palette_is_distinct_and_named():
    pal = _lib.render_palette()
    assert pal.shape == (len(_lib.RENDER_COLOURS), 3) and pal.dtype == np.uint8
    assert len({tuple(c) for c in pal}) == len(pal)
    L = _lib.load()
    assert L.msv_render_palette(None, 0) == len(pal)
    assert L.msv_render_palette(None, 1) < 0                       # a buffer is needed for a colour


def test_agent_at_origin():
    s = _empty_state(REC)
    _agent(s, 0, 0, 0)
    img = _draw(s)
    c = N_PX // 2
    _, xs, _ = rr.pixel_centres(REC, N_PX, N_PX)
    assert xs[c] == 0 and img[c, c] == rr.TICK                      # the heading tick (pointing +y) starts there
    assert img[c + 2, c] == rr.AGENT0 and img[c, c + 2] == rr.AGENT0
    r = f32(REC['agent_size'] / 2)
    past = c + int(np.argmax(xs[c:] > r))                           # first pixel centre right of agent_r
    assert img[c, past - 1] == rr.AGENT0 and img[c, past] == rr.FLOOR


def test_box_corners():
    s = _empty_state(REC)
    s['n_boxes'] = 1
    s['box_x'][0], s['box_y'][0] = f32(2.0), f32(-1.0)
    s['box_shape'][0]['hx'], s['box_shape'][0]['hy'] = f32(0.9), f32(0.5)
    img = _draw(s)
    _, xs, ys = rr.pixel_centres(REC, N_PX, N_PX)
    cols = np.nonzero(np.abs(xs - f32(2.0)) <= f32(0.9))[0]
    rows = np.nonzero(np.abs(ys - f32(-1.0)) <= f32(0.5))[0]
    for j in (rows[0], rows[-1]):
        for i in (cols[0], cols[-1]):
            assert img[j, i] == rr.BOX
    assert img[rows[0] - 1, cols[0]] == rr.FLOOR and img[rows[-1] + 1, cols[-1]] == rr.FLOOR
    assert img[rows[0], cols[0] - 1] == rr.FLOOR and img[rows[-1], cols[-1] + 1] == rr.FLOOR


def test_zone_tint_on_both_sides_of_r():
    s = _empty_state(REC)
    s['zone_cur_r'] = f32(5.0)
    img = _draw(s)
    c = N_PX // 2
    sz, xs, _ = rr.pixel_centres(REC, N_PX, N_PX)
    inside = int(np.nonzero(xs < f32(5.0) - sz)[0][-1])
    outside = int(np.nonzero(xs > f32(5.0) + sz)[0][0])
    assert img[c, inside - 1] == rr.FLOOR and img[c, outside + 1] == rr.OUTSIDE
    assert (img[c, inside + 1:outside] == rr.RING).all()
    assert img[0, 0] == rr.BG                                        # the tint stays on the floor


def test_next_zone_ring():
    s = _empty_state(REC)
    s['zone_phase'] = 0
    s['zone_cx'][1], s['zone_cy'][1] = f32(0), f32(0)
    img = _draw(s)
    R = f32(REC['zone_radiuses'][1])
    c = N_PX // 2
    assert img[c, _col(REC, N_PX, R)] == rr.NEXT_RING and img[c, c] == rr.FLOOR


def test_painter_order_agent_over_heal_over_floor():
    s = _empty_state(REC)
    s['n_heals'] = 1
    s['heal_x'][0], s['heal_y'][0] = f32(-0.4), f32(0)
    _agent(s, 0, 0.1, 0)
    img = _draw(s)
    c = N_PX // 2
    assert img[c, _col(REC, N_PX, -0.2)] == rr.AGENT0               # agent over the heal (0.2 from its centre)
    assert img[c, _col(REC, N_PX, -0.6)] == rr.HEAL                 # 0.7 from the agent's centre
    assert img[c, _col(REC, N_PX, -1.6)] == rr.FLOOR


def test_dead_agent_is_invisible():
    s = _empty_state(REC)
    _agent(s, 1, 2.0, 2.0)
    s['alive'][1] = 0
    assert (_draw(s) == _draw(_empty_state(REC))).all()


def test_heading_tick_end_point():
    s = _empty_state(REC)
    _agent(s, 0, 0, 0, angle=0.0)
    img = _draw(s)
    c = N_PX // 2
    sz, xs, _ = rr.pixel_centres(REC, N_PX, N_PX)
    r = f32(REC['agent_size'] / 2)
    w = max(sz, f32(0.2) * r)
    tip = [i for i in range(c, N_PX) if xs[i] > r]
    assert img[c, tip[0]] == rr.TICK and xs[tip[0]] - r <= w        # just past the agent: the tick
    beyond = [i for i in tip if xs[i] - r > w]
    assert img[c, beyond[0]] == rr.FLOOR
    assert img[c + 2, c] == rr.AGENT0                                 # the tick points along +x only


def test_lidar_segment_stops_at_frac():
    rec = oc.lidar_config(1, 1, 0.1, 10.0)
    s = _empty_state(rec)
    _agent(s, 0, 0, 0, angle=0.0)
    frac = np.array([[0.5]], dtype=np.float32)
    img = _draw(s, rec, frac=frac)
    c = N_PX // 2
    assert img[c, _col(rec, N_PX, 4.9)] == rr.RAY
    assert img[c, _col(rec, N_PX, 5.4)] == rr.FLOOR
    assert (_draw(s, rec) != rr.RAY).all()                            # no rays without the flag


def test_viewport_1x1_and_7x5():
    F = float(REC['floor_size'])
    V = f32(F / 2 + F / 100)
    s1, xs, ys = rr.pixel_centres(REC, 1, 1)
    assert s1 == f32(2.0) * V and xs[0] == 0 and ys[0] == 0
    s = _empty_state(REC)
    assert _draw(s, n=1)[0, 0] == rr.FLOOR
    sz, xs, ys = rr.pixel_centres(REC, 5, 7)                          # H = 5, W = 7: s from the short side
    assert sz == (f32(2.0) * V) / f32(5)
    assert list(xs) == [(f32(2 * i - 7 + 1) * f32(0.5)) * sz for i in range(7)]
    assert list(ys) == [(f32(5 - 1 - 2 * j) * f32(0.5)) * sz for j in range(5)]
    img = rr.render_indices(REC, s, 5, 7)
    assert (img[:, 0] == rr.BG).all() and (img[:, 6] == rr.BG).all()   # x = -+3s lies beyond the walls
    assert (img[:, 1:6] == rr.FLOOR).all()


def test_png_round_trip(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, 'gym-ma-survival-2d_b200'))
    import demo
    rng = np.random.default_rng(3)
    for h, w in ((1, 1), (5, 7), (33, 64)):
        img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        p = tmp_path / f'x{h}_{w}.png'
        demo.write_png(str(p), img)
        assert np.array_equal(rr.read_png(str(p)), img)
