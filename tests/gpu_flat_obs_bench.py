"""What the flat observation layout saves a trainer whose policy reads one [N, A, D] tensor.
Workloads: 2v2 at 16 384 environments, ffa at 8 192, ffa_lidar at 32 768, each handle pre-rolled --preroll
steps (episodes at their stationary mix), random actions from a fixed pool, auto-reset.  Per workload, with a
dict handle and a flat handle stepping the same actions, in --rounds rounds that alternate the arms:
  (a) a dict step followed by the trainer's flatten: torch.cat of the reshaped keys into a preallocated
      [N, A, D] tensor (out=),
  (b) a flat step (the library writes [N, A, D] itself),
  (c) k_obs2 alone in each layout, from the library's kernel timing (CUDA events around each kernel of a step;
      the tile hand-off is off while it records).
Times are CUDA events over --steps steps per round; the median of the rounds is reported.  Prints the card's
name and power limit, then one JSON line per workload.

    python tests/gpu_flat_obs_bench.py [--steps 200] [--rounds 7] [--preroll 600] [--out DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'gym-ma-survival-2d_b200'))
WORKLOADS = [('2v2', 16384), ('ffa', 8192), ('ffa_lidar', 32768)]


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def _time(fn, steps):
    import torch
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for t in range(steps):
        fn(t)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def main():
    import torch
    from masurvival.config import variant
    from masurvival.envs import MaSurvivalVec
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--preroll', type=int, default=600)
    ap.add_argument('--out', help='directory for flat_obs_bench.json')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    gpu = card()
    print('card:', gpu)
    rows = []
    for name, n in WORKLOADS:
        ed = MaSurvivalVec(variant(name), n, seed=1, obs_layout='dict')
        ef = MaSurvivalVec(variant(name), n, seed=1, obs_layout='flat')
        A = ed.n_agents
        keys = [k for k in ed.obs_shapes() if k != 'lidar_hit']
        g = torch.Generator(device='cuda'); g.manual_seed(0)
        pool = []
        for _ in range(16):
            a = torch.empty((n, A, 6), dtype=torch.uint8, device='cuda')
            a[..., :3] = torch.randint(0, 3, (n, A, 3), dtype=torch.uint8, device='cuda', generator=g)
            a[..., 3:] = torch.randint(0, 2, (n, A, 3), dtype=torch.uint8, device='cuda', generator=g)
            pool.append(a)
        ed.reset(); ef.reset()
        for t in range(args.preroll):
            ed.step(pool[t % 16]); ef.step(pool[t % 16])
        D = ef.flat_obs().shape[2]
        buf = torch.empty((n, A, D), dtype=torch.float32, device='cuda')

        def dict_and_cat(t):
            obs = ed.step(pool[t % 16])[0]
            torch.cat([obs[k].reshape(n, A, -1) for k in keys], 2, out=buf)

        def flat(t):
            ef.step(pool[t % 16])

        def dict_only(t):
            ed.step(pool[t % 16])

        dict_and_cat(0); flat(0); dict_only(0)                     # warm-up of the flatten's shapes
        ta, tb, td, oa, ob = [], [], [], [], []
        for r in range(args.rounds):
            ta.append(_time(dict_and_cat, args.steps))
            tb.append(_time(flat, args.steps))
            td.append(_time(dict_only, args.steps))
            for env, out in ((ed, oa), (ef, ob)):
                env._h.kernel_timing(True)
                for t in range(args.steps):
                    env.step(pool[t % 16])
                ms, _ = env._h.kernel_timing(False)
                out.append(ms[1])
        med = statistics.median
        row = {'workload': name, 'num_envs': n, 'D': D, 'card': gpu,
               'dict_step_plus_cat_ms': round(med(ta), 4), 'flat_step_ms': round(med(tb), 4),
               'dict_step_ms': round(med(td), 4),
               'k_obs2_dict_ms': round(med(oa), 4), 'k_obs2_flat_ms': round(med(ob), 4),
               'obs_bytes_per_env_dict': ed.obs_bytes_per_env(), 'obs_bytes_per_env_flat': ef.obs_bytes_per_env(),
               'flat_saves_ms': round(med(ta) - med(tb), 4),
               'spread_ms': {'a': [round(min(ta), 4), round(max(ta), 4)], 'b': [round(min(tb), 4), round(max(tb), 4)]}}
        print(json.dumps(row), flush=True)
        rows.append(row)
        ed.close(); ef.close()
        del pool, buf
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'flat_obs_bench.json'), 'w') as f:
            json.dump({'card': gpu, 'rows': rows}, f, indent=1)


if __name__ == '__main__':
    main()
