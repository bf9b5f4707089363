"""What the global-state output costs a step, and what it saves a trainer that would otherwise build the row itself.
Workloads: 2v2 at 16 384 environments, ffa at 8 192, ffa_lidar at 32 768, each handle pre-rolled --preroll steps
(episodes at their stationary mix), random actions from a fixed pool, auto-reset.  Per workload, with a handle
without and a handle with the output stepping the same actions, in --rounds rounds that alternate the arms:
  (a) a step with the output off,
  (b) a step with it on (k_global_state writes the [N, Ds] row after the observation kernels),
  (c) for comparison, a step of the handle of (a) (the shipped variants are omniscient) followed by the torch.cat
      a trainer would write to build the same row from the observation dict into a preallocated [N, Ds] tensor
      (out=): observer 0's copy of the per-env keys, the per-agent inventory keys, an alive mask from the agent
      rows' health column and a step counter of its own.
Times are CUDA events over --steps steps per round; the median of the rounds is reported.  Prints the card's
name and power limit, then one JSON line per workload.

    python tests/gpu_global_state_bench.py [--steps 200] [--rounds 7] [--preroll 600] [--out DIR]
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


def row_pieces(env, obs, alive_col, steps):
    """the trainer's restatement of the global-state row from an omniscient observation dict (2-D pieces)"""
    n, A = env.num_envs, env.n_agents
    agent = obs['agent']
    out = [agent.reshape(n, -1), (agent[..., alive_col] == 0).float(), obs['zone'][:, 0]]
    if env.n_heals > 0:
        out += [obs['heals'][:, 0].reshape(n, -1), obs['heals_mask'][:, 0], obs['heal_slot'].reshape(n, A),
                obs['heal_slot_mask'].reshape(n, A)]
    if env.n_boxes > 0:
        out += [obs['boxes'][:, 0].reshape(n, -1), obs['boxes_mask'][:, 0], obs['box_items'][:, 0].reshape(n, -1),
                obs['box_items_mask'][:, 0], obs['box_slot'].reshape(n, -1), obs['box_slot_mask'].reshape(n, A)]
    return out + [steps]


def main():
    import torch
    from masurvival.config import variant
    from masurvival.envs import MaSurvivalVec
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--preroll', type=int, default=600)
    ap.add_argument('--workloads', default=','.join(w for w, _ in WORKLOADS))
    ap.add_argument('--out', help='directory for global_state_bench.json')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    gpu = card()
    print('card:', gpu)
    rows = []
    for name, n in WORKLOADS:
        if name not in args.workloads.split(','):
            continue
        e0 = MaSurvivalVec(variant(name), n, seed=1)
        e1 = MaSurvivalVec(variant(name), n, seed=1, global_state=True)
        A = e0.n_agents
        g = torch.Generator(device='cuda'); g.manual_seed(0)
        pool = []
        for _ in range(16):
            a = torch.empty((n, A, 6), dtype=torch.uint8, device='cuda')
            a[..., :3] = torch.randint(0, 3, (n, A, 3), dtype=torch.uint8, device='cuda', generator=g)
            a[..., 3:] = torch.randint(0, 2, (n, A, 3), dtype=torch.uint8, device='cuda', generator=g)
            pool.append(a)
        e0.reset(); e1.reset()
        for t in range(args.preroll):
            e0.step(pool[t % 16]); e1.step(pool[t % 16])
        Ds = e1.state().shape[1]
        buf = torch.empty((n, Ds), dtype=torch.float32, device='cuda')
        steps = torch.zeros((n, 1), dtype=torch.float32, device='cuda')
        alive_col = 2 if e0.has_teams else 1      # the health column of an agent row

        def off(t):
            e0.step(pool[t % 16])

        def on(t):
            e1.step(pool[t % 16])

        def step_and_cat(t):
            obs = e0.step(pool[t % 16])[0]
            torch.cat(row_pieces(e0, obs, alive_col, steps), 1, out=buf)

        off(0); on(0); step_and_cat(0)                            # warm-up of the restatement's shapes
        ta, tb, tc = [], [], []
        for r in range(args.rounds):
            ta.append(_time(off, args.steps))
            tb.append(_time(on, args.steps))
            tc.append(_time(step_and_cat, args.steps))
        med = statistics.median
        row = {'workload': name, 'num_envs': n, 'Ds': Ds, 'card': gpu,
               'step_off_ms': round(med(ta), 4), 'step_on_ms': round(med(tb), 4),
               'step_plus_cat_ms': round(med(tc), 4),
               'on_minus_off_ms': round(med(tb) - med(ta), 4), 'cat_minus_off_ms': round(med(tc) - med(ta), 4),
               'row_bytes_per_env': 4 * Ds, 'kernel_bytes_per_env': e1._h.kernel_bytes_per_env(3),
               'spread_ms': {'a': [round(min(ta), 4), round(max(ta), 4)], 'b': [round(min(tb), 4), round(max(tb), 4)],
                             'c': [round(min(tc), 4), round(max(tc), 4)]}}
        print(json.dumps(row), flush=True)
        rows.append(row)
        e0.close(); e1.close()
        del pool, buf
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'global_state_bench.json'), 'w') as f:
            json.dump({'card': gpu, 'rows': rows}, f, indent=1)


if __name__ == '__main__':
    main()
