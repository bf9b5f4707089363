"""Quick device-side timing of the whole step (development aid; bench.py is the contract benchmark).

  python gpu_quickbench.py                      # 2v2, 16384 envs, 600 timed steps (seeded actions)
  python gpu_quickbench.py ffa 32768 300 100    # variant, envs, timed steps, warm-up steps
  python gpu_quickbench.py --sweep              # 2v2 at 1k .. 32k envs
  python gpu_quickbench.py --all                # one line per BASELINE config shape
  python gpu_quickbench.py --prof               # per-phase clock64() profile (needs `make PROFILE=1`)
MSV_LIB=/path/to/other/libmasurv.so selects another build of the library (A/B runs).
"""
import os
import sys
import parity  # noqa: F401  (puts the package and the oracle on sys.path)
from parity import make_config
import torch
from masurvival import _lib

PHASES = ['load', 'pre_step', 'find_new', 'collide', 'solve', 'toi', 'post_boxes', 'cameras', 'post_rest',
          'rewards+reset', 'observe', 'store']


BLK_PHASES = ['load', 'motors+use/give', 'melee(+find_new)', 'collide#1', 'solve#1', 'find_new#1', 'toi#1', 'collide#2', 'solve#2',
              'find_new#2', 'toi#2+box deaths', 'cameras', 'post_rest', 'rewards+reset', 'store']


def blocks(variant, N, warm=1500, launches=40):
    """per-block timeline (profile build): which phase makes the slowest block of a launch slow"""
    import ctypes
    import numpy as np
    rec = make_config(variant, auto_reset=True)
    A = int(rec['n_agents'])
    h = _lib.Handle(rec, N, 0, 1, 0)
    h.reset()
    torch.manual_seed(1234)
    NB = 61
    acts = torch.randint(0, 2, (NB, N, A, 6), dtype=torch.uint8, device='cuda')
    acts[..., 0:3] = torch.randint(0, 3, (NB, N, A, 3), dtype=torch.uint8, device='cuda')
    for t in range(warm):
        h.step(acts[(t * 7) % NB].data_ptr())
    L = _lib.load()
    L.msv_debug_profile.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    L.msv_debug_blocks.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
    L.msv_debug_profile(h.h, 1, None)
    W = 24
    buf = np.zeros(2048 * W, dtype=np.uint64)
    tot_mean, tot_max, ph_mean, ph_max, ph_maxany, toi_rows = [], [], [], [], [], []
    for t in range(launches):
        h.step(acts[((warm + t) * 7) % NB].data_ptr())
        rc = L.msv_debug_blocks(h.h, buf.ctypes.data, buf.size)
        assert rc == 0, rc
        b = buf.reshape(2048, W).astype(np.int64)
        toi_rows.append(b[2047, [0, 1, 2, 3, 4, 5, 6, 8]]); b[2047] = 0   # g_toi word 7 is unused
        nb = int((b[:, 0] > 0).sum())
        b = b[:nb]
        n = int(b[0, 0])
        d = np.diff(b[:, 1:n], axis=1)          # [blocks, phases]
        tot = d.sum(axis=1)
        k = int(tot.argmax())
        tot_mean.append(tot.mean()); tot_max.append(tot.max())
        ph_mean.append(d.mean(axis=0)); ph_max.append(d[k]); ph_maxany.append(d.max(axis=0))
        b[:, 0] = 0
    L.msv_debug_profile(h.h, 0, None)
    ph_mean, ph_max, ph_maxany = np.mean(ph_mean, axis=0), np.mean(ph_max, axis=0), np.mean(ph_maxany, axis=0)
    print(f'{variant} N={N}: {nb} blocks; block time mean {np.mean(tot_mean):.0f} cycles, slowest block of a launch {np.mean(tot_max):.0f} '
          f'(x{np.mean(tot_max) / np.mean(tot_mean):.2f}); worst launch {np.max(tot_max):.0f}, best {np.min(tot_max):.0f}')
    print('   %-20s %10s %14s %16s' % ('phase', 'mean block', 'slowest block', 'max over blocks'))
    for i in range(len(ph_mean)):
        nm = BLK_PHASES[i] if i < len(BLK_PHASES) else str(i)
        print('   %-20s %10.0f %14.0f %16.0f' % (nm, ph_mean[i], ph_max[i], ph_maxany[i]))
    print('   longest solve_toi call of each launch: cycles, loop iterations, events run, not touching, identical repeats, cycles in events, cycles in scans, env')
    for r in toi_rows[:16]:
        print('     ', ' '.join(str(int(x)) for x in r))
    h.close()


def trace(variant, N, warm=1500, launches=12):
    """hand-off trace (profile build): when do the observation tiles run relative to the step kernel's blocks"""
    import ctypes
    import numpy as np
    rec = make_config(variant, auto_reset=True)
    A = int(rec['n_agents'])
    h = _lib.Handle(rec, N, 0, 1, 0)
    h.reset()
    torch.manual_seed(1234)
    NB = 61
    acts = torch.randint(0, 2, (NB, N, A, 6), dtype=torch.uint8, device='cuda')
    acts[..., 0:3] = torch.randint(0, 3, (NB, N, A, 3), dtype=torch.uint8, device='cuda')
    for t in range(warm):
        h.step(acts[(t * 7) % NB].data_ptr())
    L = _lib.load()
    L.msv_debug_trace.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
    M = 4096
    buf = np.zeros(2 * 6 * M, dtype=np.uint64)
    L.msv_debug_trace(h.h, buf.ctypes.data, buf.size)     # clear
    for t in range(launches):
        for r in range(2):                                # two steps back to back: the trace keeps both (ticket parity)
            h.step(acts[((warm + 2 * t + r) * 7) % NB].data_ptr())
        rc = L.msv_debug_trace(h.h, buf.ctypes.data, buf.size)
        assert rc == 0, rc
        two = buf.reshape(2, 6, M).astype(np.int64)
        first = 0 if two[0, 0][two[0, 0] > 0].min() < two[1, 0][two[1, 0] > 0].min() else 1
        prev_end = None
        for b in (two[first], two[1 - first]):
            nk = int((b[0] > 0).sum()); no = int((b[2] > 0).sum())
            t0 = b[0, :nk].min()
            ks0, ks1 = b[0, :nk] - t0, b[1, :nk] - t0
            o_res, o_acq, o_done, o_stg = b[2, :no] - t0, b[3, :no] - t0, b[4, :no] - t0, b[5, :no] - t0
            kend = ks1.max()
            q = lambda x, p: float(np.percentile(x, p)) / 1e3
            gap = '' if prev_end is None else f', first block starts {(t0 - prev_end) / 1e3:+.1f} us after the previous step\'s last tile'
            print(f'{variant} N={N} launch {t}: k_step {nk} blocks, start spread {q(ks0, 100):.1f} us, block end p10/p50/p90/max = '
                  f'{q(ks1, 10):.1f}/{q(ks1, 50):.1f}/{q(ks1, 90):.1f}/{kend / 1e3:.1f} us | obs {no} tiles: resident p10/p50/p90 = '
                  f'{q(o_res, 10):.1f}/{q(o_res, 50):.1f}/{q(o_res, 90):.1f} us, acquired->staged->written median {q(o_stg - o_acq, 50):.1f} + {q(o_done - o_stg, 50):.1f} us (last 8 tiles: {q((o_stg - o_acq)[np.argsort(o_done)[-8:]], 50):.1f} + {q((o_done - o_stg)[np.argsort(o_done)[-8:]], 50):.1f}), '
                  f'written before k_step end: {int((o_done <= kend).sum())}/{no}, last tile written {(o_done.max() - kend) / 1e3:+.1f} us after k_step end{gap}')
            prev_end = t0 + o_done.max()
    h.close()


def run(variant, N, steps=600, warm=100, prof=False):
    rec = make_config(variant, auto_reset=True)
    A = int(rec['n_agents'])
    ROT = int(os.environ.get('QB_ROT', '1'))     # QB_ROT=4: four batches round-robin (working set > L2, as bench.py)
    hs = [_lib.Handle(rec, N, 0, 1 + r, r * N) for r in range(ROT)]
    h = hs[0]
    for x in hs:
        x.reset()
    torch.manual_seed(1234)   # identical action streams in every run: timing differences come from the code only
    NB = 61   # prime: every batch sees all of them in a scrambled order (see bench.py)
    acts = torch.randint(0, 2, (NB, N, A, 6), dtype=torch.uint8, device='cuda')
    acts[..., 0:3] = torch.randint(0, 3, (NB, N, A, 3), dtype=torch.uint8, device='cuda')
    # QB_STREAM=1: a non-blocking stream of our own instead of the legacy default stream
    strm = torch.cuda.Stream() if os.environ.get('QB_STREAM', '0') == '1' else torch.cuda.current_stream()
    sp = strm.cuda_stream
    torch.cuda.synchronize()
    for t in range(warm * ROT):
        hs[t % ROT].step(acts[((t // ROT) * 7 + (t % ROT) * 13) % NB].data_ptr(), sp)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(strm)
    for t in range(steps):
        hs[t % ROT].step(acts[((t // ROT) * 7 + (t % ROT) * 13) % NB].data_ptr(), sp)
    e1.record(strm)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    bps = h.bytes_per_env_step()
    st = h.flush_stats()
    tag = os.environ.get('MSV_LIB', 'default').split('/')[-1] + (' EPB=' + os.environ['MSV_EPB'] if 'MSV_EPB' in os.environ else '') + f' rot={ROT}' + (' own-stream' if sp else ' stream0') + (' NO_HANDOFF' if os.environ.get('MSV_NO_HANDOFF', '0') == '1' else '')
    print(f'[{tag}] {variant} N={N}: {ms*1e3:.1f} us/step, {N/ms*1e3:.3e} env-steps/s, {N*A/ms*1e3:.3e} agent-steps/s, '
          f'{bps} B/env-step -> {N*bps/ms/1e6:.1f} GB/s, episodes={int(st["episodes"])}')
    if prof:
        import ctypes
        L = _lib.load()
        L.msv_debug_profile.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
        buf = (ctypes.c_ulonglong * 64)()
        for x in hs:
            L.msv_debug_profile(x.h, 1, buf)
        for t in range(20 * ROT):
            hs[t % ROT].step(acts[((t // ROT) * 7 + (t % ROT) * 13) % NB].data_ptr())
        for x in hs[1:]:
            L.msv_debug_profile(x.h, 0, None)
        L.msv_debug_profile(h.h, 0, buf)
        N = N * ROT   # the sums below cover every batch
        tot = (sum(buf[:12]) + sum(buf[32:44])) or 1
        SYNCS = ['0 after load', '1 before collide', '2 before solve', '3 before toi', '4 before cameras', '5 before post_rest', '6 before melee', '7 before rewards', '8 before store_obm', '9 in solve']
        print('   slowest group (any of 20 launches): total=%d cycles, env %d; ' % (buf[12], buf[13]) + ', '.join(f'{n}={buf[16+i]}' for i, n in enumerate(PHASES)))
        print('   leader-lane cycles/env/step: ' + ', '.join(f'{n}={buf[i]/N/20:.0f} ({buf[i]/tot:.0%})' for i, n in enumerate(PHASES)))
        print('   barrier waits cycles/env/step: ' + ', '.join(f'[{n}]={buf[32+i]/N/20:.0f} ({buf[32+i]/tot:.0%})' for i, n in enumerate(SYNCS)))
        print('   slowest group waits: ' + ', '.join(f'[{n}]={buf[48+i]}' for i, n in enumerate(SYNCS)))
        print('   total cycles/env/step %.0f' % (tot / N / 20))
        rare = [('generic island solve', 44), ('TOI event', 46), ('reset', 58), ('deaths', 60), ('pickups', 62), ('use/give', 14), ('contact numbering', 42)]
        print('   rare paths (calls per 1000 env-steps, mean cycles per call): ' +
              ', '.join(f'{n}: {buf[i] / (N * 20) * 1000:.2f} x {buf[i + 1] / max(buf[i], 1):.0f}' for n, i in rare))
        nev = max(buf[46], 1)
        print('   toi_event sub-phases (mean cycles): ' + ', '.join(f'{n}={buf[20 + i] / nev:.0f}' for i, n in enumerate(
            ['advance+update', 'other contacts', 'position solve', 'velocity solve', 'integrate+sync+broadphase', 'snapshot'])))
        nis = max(buf[44], 1); ngen = max(buf[48 + 6], 1)
        print('   solve_island: DFS+damping mean %.0f; pair path mean %.0f; general path: %d calls (%.2f per 1000 env-steps), mean contacts %.1f, init %.0f, velocity %.0f, integrate+position %.0f cycles' % (
            buf[48] / nis, buf[49] / max(nis - buf[54], 1), buf[54], buf[54] / (N * 20) * 1000, buf[55] / ngen, buf[50] / ngen, buf[51] / ngen, buf[52] / ngen))
        print('   longest single sections: island_single<3> %d cycles (cnt %d), island_single<big> %d cycles (cnt %d), solve_island %d cycles (%d agents)' % (
            buf[26] >> 8, buf[26] & 255, buf[27] >> 8, buf[27] & 255, buf[53] >> 8, buf[53] & 255))
        print('   b2TimeOfImpact calls per 1000 env-steps: %.1f, mean cycles %.0f' % (buf[28] / (N * 20) * 1000, buf[31] / max(buf[28], 1)))
    for x in hs:
        x.close()


if __name__ == '__main__':
    a = sys.argv[1:]
    if a and a[0] == '--sweep':
        for N in (1024, 2048, 4096, 8192, 16384, 32768):
            run('2v2', N, steps=500)
    elif a and a[0] == '--all':
        for v, N in (('2v2', 16384), ('1v1_heal_only', 4096), ('1v1', 16384), ('ffa', 32768), ('ffa_lidar', 32768)):
            run(v, N, steps=500)
    elif a and a[0] == '--trace':
        trace(a[1] if len(a) > 1 else '2v2', int(a[2]) if len(a) > 2 else 16384)
    elif a and a[0] == '--blocks':
        blocks(a[1] if len(a) > 1 else '2v2', int(a[2]) if len(a) > 2 else 16384)
    elif a and a[0] == '--prof':
        run(a[1] if len(a) > 1 else '2v2', int(a[2]) if len(a) > 2 else 16384, steps=400, warm=1500, prof=True)   # stationary episode mix
    else:
        v = a[0] if a else '2v2'
        N = int(a[1]) if len(a) > 1 else 16384
        run(v, N, int(a[2]) if len(a) > 2 else 600, int(a[3]) if len(a) > 3 else 1500)   # default warm-up: stationary episode mix
