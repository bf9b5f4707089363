#!/usr/bin/env python
"""Headless counterpart of the reference's demo.py (demo.py:76-158, 164-293)
for the batched B200 environment: random-policy rollout, optional JSON config
(`-c`, same nested keys as the reference; shapes are given as radii), episode
statistics (`flush_stats`), the `--benchmark` per-step timing line, and a
headless frame dumper (`--dump-frames DIR`): after every `--frame-every`-th
step, a grid of the first `--frame-envs` environments drawn on the GPU
(MaSurvivalVec.render) is written as DIR/frame_<step>.png.  Frames are drawn
outside the timed window.  The pygame window and interactive play of the
reference are not reproduced.

    python gym-ma-survival-2d_b200/demo.py -n 4096 --max-steps 1000 --benchmark
    python gym-ma-survival-2d_b200/demo.py -n 16 --max-steps 200 --dump-frames frames --frame-envs 4
"""
import argparse
import json
import math
import os
import pprint
import struct
import sys
import time
import zlib

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from masurvival.envs import MaSurvivalVec  # noqa: E402


class RandomPolicy:
    """demo.py:18-22: `action_space.sample()`, here for N envs on the device."""

    def __init__(self, env, seed=0):
        import torch
        self.env, self.g = env, torch.Generator(device=f'cuda:{env.device}')
        self.g.manual_seed(seed)

    def act(self, observations=None):
        import torch
        N, A, dev = self.env.num_envs, self.env.n_agents, f'cuda:{self.env.device}'
        a = torch.empty((N, A, 6), dtype=torch.uint8, device=dev)
        a[..., :3] = torch.randint(0, 3, (N, A, 3), dtype=torch.uint8, device=dev, generator=self.g)
        a[..., 3:] = torch.randint(0, 2, (N, A, 3), dtype=torch.uint8, device=dev, generator=self.g)
        return a


def write_png(path, rgb):
    """uint8[H, W, 3] -> PNG (8-bit RGB, one zlib stream, filter type 0 on every row); standard library only."""
    h, w, _ = rgb.shape
    raw = b''.join(b'\x00' + rgb[y].tobytes() for y in range(h))

    def chunk(tag, data):
        return struct.pack('>I', len(data)) + tag + data + struct.pack('>I', zlib.crc32(tag + data) & 0xffffffff)
    with open(path, 'wb') as f:
        f.write(b'\x89PNG\r\n\x1a\n' + chunk(b'IHDR', struct.pack('>IIBBBBB', w, h, 8, 2, 0, 0, 0))
                + chunk(b'IDAT', zlib.compress(raw, 6)) + chunk(b'IEND', b''))


class FrameDumper:
    """Grid of the first `k` environments, ceil(sqrt(k)) per row, `size` pixels each: drawn and assembled
    on the device, copied to the host once per frame."""

    def __init__(self, env, out_dir, k=1, size=256, every=1):
        import torch
        if not 1 <= k <= env.num_envs:
            raise ValueError(f'--frame-envs must be in 1..{env.num_envs}')
        if every < 1:
            raise ValueError('--frame-every must be >= 1')
        self.env, self.dir, self.k, self.size, self.every = env, out_dir, k, size, every
        self.cols = math.ceil(math.sqrt(k))
        self.rows = math.ceil(k / self.cols)
        dev = f'cuda:{env.device}'
        self.frames = torch.empty((k, size, size, 3), dtype=torch.uint8, device=dev)
        self.grid = torch.zeros((self.rows * self.cols, size, size, 3), dtype=torch.uint8, device=dev)
        os.makedirs(out_dir, exist_ok=True)

    def __call__(self, t):
        if t % self.every:
            return
        self.env.render(count=self.k, height=self.size, width=self.size, out=self.frames)
        self.grid[:self.k] = self.frames
        S = self.size
        img = self.grid.view(self.rows, self.cols, S, S, 3).permute(0, 2, 1, 3, 4).reshape(self.rows * S, self.cols * S, 3)
        write_png(os.path.join(self.dir, f'frame_{t:05d}.png'), img.cpu().numpy())


def demo_env(env, max_steps=None, print_benchmark=False, seed=0, dumper=None):
    """Runs until every env finished one episode (auto_reset off) or max_steps; `dumper(t)` is called
    after step t (1, 2, ...), outside the timed window."""
    import torch
    policy = RandomPolicy(env, seed)
    times = []
    t, obs = 0, env.reset()
    done_once = torch.zeros(env.num_envs, dtype=torch.bool, device=f'cuda:{env.device}')
    while True:
        action = policy.act(obs)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        obs, reward, done, info = env.step(action)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        done_once |= done
        t += 1
        if dumper is not None:
            dumper(t)
        if max_steps is not None and t == max_steps:
            print(f'Maximum number of steps {t} reached, terminating episode.')
            break
        if max_steps is None and bool(done_once.all()):
            break
    print('Episode complete. Stats printed below.')
    pprint.PrettyPrinter().pprint(env.flush_stats())
    if print_benchmark:
        times = np.array(times)
        print(f'Performance test results: {times.mean()}, {times.std()}')
        print(f'  = {env.num_envs * env.n_agents / times.mean():.4g} agent-steps/s over {env.num_envs} envs')
    env.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('-c', '--config', help='JSON file with the (partial) nested config dict')
    ap.add_argument('-n', '--num-envs', type=int, default=1024)
    ap.add_argument('-s', '--max-steps', type=int, default=None)
    ap.add_argument('-b', '--benchmark', action='store_true', help='print mean/std of the per-step time (demo.py:274-279)')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--device', type=int, default=0)
    ap.add_argument('--dump-frames', metavar='DIR', help='write a PNG of the first --frame-envs environments after steps')
    ap.add_argument('--frame-envs', type=int, default=1, metavar='K', help='environments per frame, ceil(sqrt(K)) per row')
    ap.add_argument('--frame-size', type=int, default=256, metavar='S', help='pixels per environment (S x S)')
    ap.add_argument('--frame-every', type=int, default=1, metavar='T', help='a frame after every T-th step')
    args = ap.parse_args()
    config = None
    if args.config is not None:
        with open(args.config) as f:
            config = json.load(f)
    env = MaSurvivalVec(config, num_envs=args.num_envs, device=args.device, seed=args.seed, auto_reset=args.max_steps is not None)
    dumper = None
    if args.dump_frames is not None:
        dumper = FrameDumper(env, args.dump_frames, args.frame_envs, args.frame_size, args.frame_every)
    demo_env(env, args.max_steps, args.benchmark, args.seed, dumper)


if __name__ == '__main__':
    main()
