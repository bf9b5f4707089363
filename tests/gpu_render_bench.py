"""Time msv_render (k_render) with CUDA events, beside a step of the same batch:
  (a) 16 environments of the 2v2 workload at 256x256,
  (b) all 16 384 environments of the 2v2 workload at 64x64,
  (c) 32 768 environments of ffa_lidar at 64x64 with the lidar rays.
Prints the card's name and power limit, then one JSON line per case: render and step milliseconds (mean over
--iters launches after --warmup), bytes written, GB/s and its fraction of the 6 534 GB/s the project uses as the
HBM peak, and the render's share of a step.  Case (b) writes 201 MB per launch, more than the 126 MB L2.

    python tests/gpu_render_bench.py [--iters 200] [--warmup 20] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'gym-ma-survival-2d_b200'))
PEAK_GBS = 6534.0
CASES = [('a', '2v2', 16384, 16, 256, False), ('b', '2v2', 16384, 16384, 64, False),
         ('c', 'ffa_lidar', 32768, 32768, 64, True)]


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def _time(fn, iters, warmup):
    import torch
    for _ in range(warmup):
        fn()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def main():
    import torch
    from masurvival.config import variant
    from masurvival.envs import MaSurvivalVec
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--iters', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--out', help='directory for render_bench.json')
    args = ap.parse_args()
    if args.iters < 200:
        raise SystemExit('--iters must be >= 200')
    gpu = card()
    print('card:', gpu)
    rows = []
    for tag, name, n_envs, count, size, lidar in CASES:
        env = MaSurvivalVec(variant(name), n_envs, seed=1, auto_reset=True)
        env.reset()
        g = torch.Generator(device='cuda:0')
        g.manual_seed(1)
        acts = [torch.randint(0, 2, (n_envs, env.n_agents, 6), dtype=torch.uint8, device='cuda:0', generator=g)
                for _ in range(8)]
        for a in acts:
            a[..., :3] %= 3
        for a in acts * 8:                              # past the reset transient
            env.step(a)
        k = [0]

        def step():
            env.step(acts[k[0] % len(acts)])
            k[0] += 1
        out = torch.empty((count, size, size, 3), dtype=torch.uint8, device='cuda:0')
        step_ms = _time(step, args.iters, args.warmup)
        render_ms = _time(lambda: env.render(count=count, height=size, width=size, lidar=lidar, out=out),
                          args.iters, args.warmup)
        nbytes = count * size * size * 3
        gbs = nbytes / (render_ms * 1e-3) / 1e9
        row = {'case': tag, 'workload': name, 'envs': n_envs, 'rendered': count, 'size': size, 'lidar': lidar,
               'render_ms': round(render_ms, 5), 'step_ms': round(step_ms, 5), 'bytes': nbytes,
               'GBps': round(gbs, 1), 'frac_of_peak': round(gbs / PEAK_GBS, 4),
               'share_of_step': round(render_ms / step_ms, 4), 'card': gpu}
        print(json.dumps(row), flush=True)
        rows.append(row)
        env.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'render_bench.json'), 'w') as f:
            json.dump(rows, f, indent=1)


if __name__ == '__main__':
    main()
