"""numpy float32 restatement of msv_render's picture (include/masurv.h, csrc/msv_render.cu header), drawn from
an msv_env_state record and the packed config.  It shares no code with the kernel: layers are painted bottom-up
over whole-image arrays, where the kernel searches the layers top-down per pixel.  Every expression is the
kernel's float32 expression in the same order (the library builds with -fmad=false), so the two agree bit for
bit.  Colours come from the library's table (msv_render_palette, no device needed).

The picture: viewport half-width V = (float)(F/2 + F/100), pixel size s = 2V / min(W, H), pixel centres
x = ((float)(2i - W + 1) * 0.5f) * s, y = ((float)(H - 1 - 2j) * 0.5f) * s (row 0 at the top).  Layers, later on
top: background; floor |x|, |y| <= F/2; the floor outside the current zone (d2 > r*r); the current zone's ring and
then the next zone's (lo*lo <= d2 <= hi*hi, lo = max(R - s, 0), hi = R + s; the next zone only while
phase < zone_phases - 1); the walls as axis-aligned rectangles (their float rotation of (float)(pi/2) ignored);
heals; box items (circles of the item radius); boxes (rectangles); living agents in index order; their heading
ticks (segment to centre + agent_r * (cos, sin), half-width max(s, 0.2 * agent_r)); with the lidar flag every
living agent's rays (segment to centre + frac * off, half-width 0.5 * s).  A body smaller than a pixel may cover
no pixel centre and then does not show."""
import math
import struct
import zlib

import numpy as np

f32 = np.float32
(BG, FLOOR, OUTSIDE, RING, NEXT_RING, WALL, HEAL, ITEM, BOX) = range(9)
AGENT0, TEAM0, TEAM1, TICK, RAY = 9, 17, 18, 19, 20


def palette():
    from masurvival import _lib
    return _lib.render_palette()


def pixel_centres(rec, H, W):
    """(s, xs[W], ys[H]) of an H x W image"""
    F = float(rec['floor_size'])
    V = f32(F / 2 + F / 100)
    s = (f32(2.0) * V) / f32(min(W, H))
    xs = (np.arange(W).astype(np.int64) * 2 - W + 1).astype(np.float32) * f32(0.5) * s
    ys = (H - 1 - 2 * np.arange(H).astype(np.int64)).astype(np.float32) * f32(0.5) * s
    return s, xs.astype(np.float32), ys.astype(np.float32)


def sincos(angle):
    """b2Rot::Set: sin and cos of a float angle evaluated in double, rounded to float"""
    a = float(f32(angle))
    return f32(math.sin(a)), f32(math.cos(a))


def _segment(X, Y, px, py, ex, ey, w):
    dx, dy = X - px, Y - py
    len2 = ex * ex + ey * ey
    if len2 != f32(0):
        t = np.fmin(np.fmax((dx * ex + dy * ey) / len2, f32(0)), f32(1))
    else:
        t = f32(0)
    qx, qy = dx - t * ex, dy - t * ey
    return qx * qx + qy * qy <= w * w


def render_reference(rec, s_, H, W, lidar_frac=None):
    """uint8[H, W, 3] picture of environment state `s_` (an msv_env_state record) of config `rec`;
    lidar_frac: the environment's float32[A, L] lidar_frac rows to draw the rays, or None"""
    return palette()[render_indices(rec, s_, H, W, lidar_frac)]


def render_indices(rec, s_, H, W, lidar_frac=None):
    """the same picture as palette indices, int[H, W]"""
    F = float(rec['floor_size'])
    A = int(rec['n_agents'])
    s, xs, ys = pixel_centres(rec, H, W)
    X, Y = np.meshgrid(xs, ys)
    out = np.full((H, W), BG, dtype=np.int64)
    hf = f32(F / 2)
    on_floor = (np.abs(X) <= hf) & (np.abs(Y) <= hf)
    out[on_floor] = FLOOR

    def d2(cx, cy):
        dx, dy = X - f32(cx), Y - f32(cy)
        return dx * dx + dy * dy

    zr = f32(s_['zone_cur_r'])
    out[on_floor & (d2(s_['zone_cur_x'], s_['zone_cur_y']) > zr * zr)] = OUTSIDE
    rings = [(s_['zone_cur_x'], s_['zone_cur_y'], zr, RING)]
    ph = int(s_['zone_phase'])
    if ph < int(rec['zone_phases']) - 1:
        nr = int(rec['zone_n_radiuses'])
        R = f32(rec['zone_radiuses'][ph + 1]) if ph + 1 < nr else f32(0)
        rings.append((s_['zone_cx'][ph + 1], s_['zone_cy'][ph + 1], R, NEXT_RING))
    for cx, cy, R, col in rings:
        lo, hi = max(f32(R) - s, f32(0)), f32(R) + s
        d = d2(cx, cy)
        out[(lo * lo <= d) & (d <= hi * hi)] = col
    o = f32(F / 2)
    whx, why = f32((F / 100) / 2.), f32(F / 2.)
    for cx, cy, hx, hy in ((-o, f32(0), whx, why), (f32(0), o, why, whx), (o, f32(0), whx, why), (f32(0), -o, why, whx)):
        out[(np.abs(X - cx) <= hx) & (np.abs(Y - cy) <= hy)] = WALL
    heal_r, item_r, agent_r = f32(rec['heal_item_size'] / 2), f32(rec['box_item_size'] / 2), f32(rec['agent_size'] / 2)
    for k in range(int(s_['n_heals'])):
        out[d2(s_['heal_x'][k], s_['heal_y'][k]) <= heal_r * heal_r] = HEAL
    for k in range(int(s_['n_items'])):
        out[d2(s_['item_x'][k], s_['item_y'][k]) <= item_r * item_r] = ITEM
    for k in range(int(s_['n_boxes'])):
        cx, cy = f32(s_['box_x'][k]), f32(s_['box_y'][k])
        hx, hy = f32(s_['box_shape'][k]['hx']), f32(s_['box_shape'][k]['hy'])
        out[(np.abs(X - cx) <= hx) & (np.abs(Y - cy) <= hy)] = BOX
    alive = [i for i in range(A) if s_['alive'][i]]
    for i in alive:
        col = (TEAM0 if i < A // 2 else TEAM1) if rec['teams'] else AGENT0 + i
        out[d2(s_['x'][i], s_['y'][i]) <= agent_r * agent_r] = col
    w_tick = max(s, f32(0.2) * agent_r)
    for i in alive:
        x, y = f32(s_['x'][i]), f32(s_['y'][i])
        sn, cs = sincos(s_['angle'][i])
        ex, ey = (x + agent_r * cs) - x, (y + agent_r * sn) - y
        out[_segment(X, Y, x, y, ex, ey, w_tick)] = TICK
    if lidar_frac is not None:
        L, fov, depth = int(rec['lidar_n']), float(rec['lidar_fov']), f32(rec['lidar_depth'])
        angs = [r * (fov / (L - 1)) - fov / 2. if L > 1 else 0.0 for r in range(L)]
        w_ray = f32(0.5) * s
        for i in alive:
            x, y = f32(s_['x'][i]), f32(s_['y'][i])
            for r in range(L):
                sn, cs = sincos(f32(angs[r] + float(f32(s_['angle'][i]))))
                offx, offy = cs * depth + (-sn) * f32(0), sn * depth + cs * f32(0)
                fr = f32(lidar_frac[i][r])
                ex, ey = (x + fr * offx) - x, (y + fr * offy) - y
                out[_segment(X, Y, x, y, ex, ey, w_ray)] = RAY
    return out


def read_png(path):
    """decode an 8-bit RGB PNG of filter type 0 (what demo.py writes) to uint8[H, W, 3], checking every CRC"""
    data = open(path, 'rb').read()
    assert data[:8] == b'\x89PNG\r\n\x1a\n'
    pos, chunks = 8, {}
    while pos < len(data):
        n, = struct.unpack('>I', data[pos:pos + 4])
        tag, body = data[pos + 4:pos + 8], data[pos + 8:pos + 8 + n]
        crc, = struct.unpack('>I', data[pos + 8 + n:pos + 12 + n])
        assert crc == zlib.crc32(tag + body) & 0xffffffff
        chunks[tag] = chunks.get(tag, b'') + body
        pos += 12 + n
    w, h, depth, ctype, _, _, _ = struct.unpack('>IIBBBBB', chunks[b'IHDR'])
    assert depth == 8 and ctype == 2 and b'IEND' in chunks
    raw = zlib.decompress(chunks[b'IDAT'])
    rows = [raw[y * (3 * w + 1):(y + 1) * (3 * w + 1)] for y in range(h)]
    assert all(r[0] == 0 for r in rows)                               # filter type 0
    return np.frombuffer(b''.join(r[1:] for r in rows), dtype=np.uint8).reshape(h, w, 3)
