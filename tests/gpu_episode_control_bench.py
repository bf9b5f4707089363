"""Cost of the step limit, of terminal capture and of msv_reset_envs on the 2v2 workload (16 384 environments).
  (a) ms per step with auto_reset=True and max_episode_steps T = 0, 300 and 10**6, and with auto_reset='terminal'
      and T = 0 and 300.  The five handles are pre-rolled to the stationary episode mix (--preroll steps each, as
      bench.py does) and timed in alternating blocks of --steps steps (CUDA events around each block); the median
      block over --rounds rounds is reported.  auto_reset=True with T = 0 runs the tile hand-off; the other cases
      give it up and add k_truncate (T > 0), the row-filtered k_obs2 into terminal_* (terminal) and the k_reset
      of the finished environments.
  (b) device-event time of one reset_envs with 1 %, 10 % and 100 % of the environments masked (mean over --iters
      calls, one untimed step between calls).
Each handle's state and outputs (about 100 MB) largely fit the 126 MB L2, unlike bench.py's rotating batches.
Prints the card's name and power limit, then one JSON line per case.

    python tests/gpu_episode_control_bench.py [--preroll 1500] [--steps 200] [--rounds 7] [--iters 100] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'gym-ma-survival-2d_b200'))
N = 16384


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def main():
    import numpy as np
    import torch
    from masurvival.config import variant
    from masurvival.envs import MaSurvivalVec
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--preroll', type=int, default=1500)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--iters', type=int, default=100)
    ap.add_argument('--out', help='directory for episode_control_bench.json')
    args = ap.parse_args()
    gpu = card()
    print('card:', gpu, flush=True)
    g = torch.Generator(device='cuda:0')
    g.manual_seed(1)
    acts = [torch.randint(0, 2, (N, 4, 6), dtype=torch.uint8, device='cuda:0', generator=g) for _ in range(16)]
    for a in acts:
        a[..., :3] = torch.randint(0, 3, (N, 4, 3), dtype=torch.uint8, device='cuda:0', generator=g)
    cases = ((True, 0), (True, 300), (True, 10 ** 6), ('terminal', 0), ('terminal', 300))    # (auto_reset, T)
    envs = {c: MaSurvivalVec(variant('2v2'), N, seed=1, auto_reset=c[0], max_episode_steps=c[1]) for c in cases}
    k = {c: 0 for c in cases}

    def step(c):
        envs[c].step(acts[k[c] % len(acts)])
        k[c] += 1
    for c in cases:
        envs[c].reset()
        for _ in range(args.preroll):
            step(c)
    torch.cuda.synchronize()
    blocks = {c: [] for c in cases}
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for c in cases:
            t0.record()
            for _ in range(args.steps):
                step(c)
            t1.record()
            torch.cuda.synchronize()
            blocks[c].append(t0.elapsed_time(t1) / args.steps)
    rows = []
    for c in cases:
        b = sorted(blocks[c])
        row = {'case': 'step', 'workload': '2v2', 'envs': N, 'auto_reset': c[0], 'max_episode_steps': c[1],
               'ms_per_step': round(b[len(b) // 2], 5), 'min': round(b[0], 5), 'max': round(b[-1], 5), 'blocks': len(b),
               'steps_per_block': args.steps, 'hand_off': envs[c].tile_plan()['observation_hand_off'], 'card': gpu}
        print(json.dumps(row), flush=True)
        rows.append(row)
    env = envs[(True, 0)]
    rng = np.random.default_rng(2)
    for frac in (0.01, 0.10, 1.0):
        mask = torch.as_tensor(rng.random(N) < frac if frac < 1 else np.ones(N, bool)).cuda()
        tot = 0.0
        for i in range(args.iters + 5):
            step((True, 0))
            t0.record()
            env.reset_envs(mask)
            t1.record()
            torch.cuda.synchronize()
            if i >= 5:                                     # warm-up
                tot += t0.elapsed_time(t1)
        row = {'case': 'reset_envs', 'workload': '2v2', 'envs': N, 'masked': int(mask.sum()), 'fraction': frac,
               'ms': round(tot / args.iters, 5), 'iters': args.iters, 'card': gpu}
        print(json.dumps(row), flush=True)
        rows.append(row)
    for e in envs.values():
        e.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'episode_control_bench.json'), 'w') as f:
            json.dump(rows, f, indent=1)


if __name__ == '__main__':
    main()
