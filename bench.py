#!/usr/bin/env python
"""bench.py -- headline benchmark of the masurvival step path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload 2v2|1v1_heal_only|ffa|ffa_lidar] [--dump-outputs DIR]

Default workload = BASELINE.json configs[2], the config the metric is quoted on:
default 2v2 (A=4, teams, melee cd 40, B=4, H=4, shrinking safe zone), 16384
environments PER GPU, random actions, auto-reset.  One "step" = one
MaSurvival.step of every environment of the batch.  Environments shard
trivially: one process per GPU, no collective on the data path (SURVEY.md
section 8e) -> weak scaling.

What is timed is the STATIONARY workload, whatever --steps/--warmup are: before
the timed region every batch is pre-rolled `--preroll` (default 1500) untimed
steps so that episode phases are de-synchronised (mean episode ~420 steps) and
contacts, TOI events, melee hits, deaths, death-drops and in-kernel auto-resets
all occur at their steady-state rates.  Then a fixed number of untimed steps
that keep the device busy, W warm-up steps, and EXACTLY K timed steps: up to
--repeats repeats of >= 20 steps, spread over 3 000 steps of the roll-out
with untimed steps between them (the step time drifts over a few hundred
steps), each bracketed by barrier + synchronize and timed with CUDA events,
MAX over ranks per repeat; `ms_per_step` is the MEDIAN per-step time of the
repeats.  Every step count depends on the arguments alone, so the same
arguments give the same inputs on every run and every build.

`--dump-outputs DIR` writes what the last timed step returned (observation
tensors in the library's layout, rewards, dones, episode statistics) as
DIR/<name>.npy in float32, for the environments listed in env_index.npy: all
of them, or a fixed seeded sample that keeps the files under 64 MB.  Two
builds run with the same arguments can be compared output for output.

Prints ONE JSON line (rank 0).  `value` = agent-steps/s with actions already
resident in HBM; `e2e` = the same through the host-buffer C-ABI call
(H2D actions + D2H rewards/dones inside the timed region), `e2e_obs` with the
observation tensors copied back as well.  `--impl reference` times the CPU
oracle port (the reference's own pybox2d stack is not installable here,
DESIGN.md) on all host threads, same pre-roll, same config block.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, 'gym-ma-survival-2d_b200'))

METRIC = 'agent_steps_per_sec'
UNIT = 'agent-steps/s'
L2_BYTES = 126e6
NB_CPU = 61   # pre-generated random action batches of the CPU arms (same cycling rule as the GPU arm)
BUSY_STEPS = 2500      # untimed steps right before the timed repeats: >= 150 ms of work for every workload below on a B200
SPAN_STEPS = 3000      # the timed repeats are spread over this many steps of the roll-out (see run_ours)
MIN_REPEAT_STEPS = 20  # shorter repeats would time the barrier around them as much as the steps
DUMP_BYTES = 64 << 20  # --dump-outputs: at most this many bytes of .npy files

# BASELINE.json `configs` made concrete (SURVEY.md section 8d / BASELINE.md section 3).  `rotate`: independent
# batches stepped round-robin so that their state + outputs exceed the 126 MB L2 (1.3x L2 over the library's
# device bytes per batch); fixed here rather than derived from the build, so every build steps the same batches.
WORKLOADS = {
    '2v2': dict(variant='2v2', envs=16384, agents=4, rotate=3, kernel='k_step<4,4,4,4>',
                label='configs[2]: default 2v2 (A=4 teams, melee cd40, B=4, H=4, safe zone), random actions, auto-reset'),
    '1v1_heal_only': dict(variant='1v1_heal_only', envs=4096, agents=2, rotate=23, kernel='k_step<2,4,4,2>',
                          label='configs[1]: 1v1 heal-only (A=2, B=0, H=4, melee damage 0), random actions, auto-reset'),
    'ffa': dict(variant='ffa', envs=8192, agents=8, rotate=3, kernel='k_step<8,8,16,8>',
                label='configs[3]: free-for-all max (A=8, B=8 randomized, H=16, grid 8), 65536 envs across 8 GPUs = 8192 per GPU, auto-reset'),
    'ffa_lidar': dict(variant='ffa_lidar', envs=32768, agents=8, rotate=2, kernel='k_step<8,8,16,8>',
                      label='configs[4]: ffa max + 32-ray lidar block (doubled rays), 32768 envs per GPU, auto-reset'),
}


def repeat_sizes(k, r):
    """K timed steps as at most r repeats of >= MIN_REPEAT_STEPS steps (one if K is smaller), lengths within one"""
    r = max(1, min(r, k // MIN_REPEAT_STEPS))
    return [k // r + (i < k % r) for i in range(r)]


def dump_sample(n, bytes_per_env, n_files):
    """environments written by --dump-outputs: all n, or a fixed seeded sample that keeps n_files .npy files
    (128-byte headers) within DUMP_BYTES"""
    cap = max(1, (DUMP_BYTES - 128 * n_files) // bytes_per_env)
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, size=cap, replace=False))


def write_dump(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), np.ascontiguousarray(a, dtype=np.float32))


def workload_config(name, auto_reset=True):
    from masurvival.config import merge_config, pack_config, variant
    cfg, cm = merge_config(variant(WORKLOADS[name]['variant']))
    return pack_config(cfg, cm, auto_reset=auto_reset)


def config_block(name, n_gpus, envs_per_gpu):
    w = WORKLOADS[name]
    return {'workload': w['label'], 'envs_per_gpu': envs_per_gpu, 'global_envs': envs_per_gpu * n_gpus,
            'agents_per_env': w['agents'],
            'parallelism': f'{n_gpus} independent env shards (1 process/GPU, no collective)'}


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def ncu_counters(name):
    """per-launch counters of the dominant kernel from the committed ncu --set full capture
    (profiles/counters.json): DRAM traffic and warp instructions; None when not captured"""
    p = os.path.join(ROOT, 'profiles', 'counters.json')
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(name, {})
        except Exception:
            return {}
    return {}


def ref_python_baseline(name):
    """`ref-python-on-shim` (BASELINE.md section 3): the reference's unmodified Python on the
    Box2D/gym shims.  /root/reference does not exist on the GPU box, so this is the figure
    measured in the build container by tests/golden/time_reference.py (committed)."""
    p = os.path.join(ROOT, 'profiles', 'ref_python_on_shim.json')
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(name)
        except Exception:
            return None
    return None


class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu):
        self.gpu, self.p = gpu, None

    def start(self):
        try:
            self.p = subprocess.Popen(['nvidia-smi', f'--id={self.gpu}', f'--query-gpu={self.Q}',
                                       '--format=csv,noheader,nounits', '-lms', '50'],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.12)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill(); out = ''
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from masurvival.envs import MaSurvivalVec
    from masurvival.config import variant

    W = WORKLOADS[args.workload]
    rank = int(os.environ.get('RANK', 0)); world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the product has no CPU fallback')
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device(f'cuda:{local}'))
    n_gpus = world
    N, A = args.envs or W['envs'], W['agents']
    dev = f'cuda:{local}'

    def make_env(r):
        return MaSurvivalVec(variant(W['variant']), num_envs=N, device=local, seed=args.seed + r,
                             env_offset=(rank * 64 + r) * N, auto_reset=True)

    # ROT independent batches of N envs are stepped round-robin: their combined state + outputs
    # exceed the 126 MB L2, so every step finds its data in HBM (timing rule: "inputs larger
    # than L2") and no flush kernel perturbs the timed region.
    envs = [make_env(0)]
    batch_bytes = envs[0].device_bytes()
    ROT = args.rotate or int(min(32, max(2, math.ceil(W['rotate'] * W['envs'] / N))))
    envs += [make_env(r) for r in range(1, ROT)]
    for e_ in envs:
        e_.reset()
    env = envs[0]
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    # Random policy (demo.py:18-22: action_space.sample() every step).  NB pre-generated action batches;
    # batch r's k-th step uses batch (k * 7 + r * 13) mod NB with NB prime, so every env sees all NB
    # batches in a scrambled order before any repeats (a short cycle would act like a constant drift:
    # agents pile into the walls and the contact/TOI rates are no longer those of a random policy).
    NB = 61

    acts_dev = torch.empty((NB, N, A, 6), dtype=torch.uint8, device=dev)
    acts_dev[..., 0:3] = torch.randint(0, 3, (NB, N, A, 3), dtype=torch.uint8, device=dev, generator=g)
    acts_dev[..., 3:6] = torch.randint(0, 2, (NB, N, A, 3), dtype=torch.uint8, device=dev, generator=g)
    acts_host = acts_dev.cpu().pin_memory()
    rew_host = [torch.empty((N, A), dtype=torch.float32).pin_memory() for _ in range(ROT)]
    done_host = [torch.empty((N,), dtype=torch.uint8).pin_memory() for _ in range(ROT)]
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            tt = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())
        return ms

    tick = [0]

    def abatch(t):
        return ((t // ROT) * 7 + (t % ROT) * 13) % NB

    def dev_step():
        t = tick[0]; tick[0] += 1
        envs[t % ROT]._h.step(acts_dev[abatch(t)].data_ptr(), stream)

    def timed(fn, k):
        """K calls of fn between barrier+synchronize, CUDA events on the launch stream, max over ranks"""
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0.record()
        for _ in range(k):
            fn()
        t1.record()
        barrier()
        return max_over_ranks(float(t0.elapsed_time(t1)))

    # ---- episode-phase profile: ms/step right after a synchronised reset (all envs at the same
    # episode step), before the pre-roll de-synchronises them -----------------------------------
    phase_ms = {}
    if not args.no_phase:
        marks = [(0, 50, 'steps 0-50 (post-reset transient)'), (150, 200, 'steps 150-200'), (350, 400, 'steps 350-400'), (700, 750, 'steps 700-750')]
        t_ep = 0
        for lo, hi, label in marks:
            for _ in range((lo - t_ep) * ROT):
                dev_step()
            phase_ms[label] = timed(dev_step, (hi - lo) * ROT) / ((hi - lo) * ROT)
            t_ep = hi
        preroll_left = max(0, args.preroll - t_ep)
    else:
        preroll_left = args.preroll
    # ---- pre-roll to the stationary episode mix ------------------------------------------------
    for _ in range(preroll_left * ROT):
        dev_step()
    torch.cuda.synchronize()
    st0 = [e_.flush_stats() for e_ in envs]   # zero the accumulators: stats below describe the timed region only

    # ---- device-resident arm -------------------------------------------------------------------
    clk = ClockSampler(local)
    if not os.environ.get('BENCH_NO_SMI'):
        clk.start()
    # The host-side pauses above (stats read-back, sampler start) let the GPU idle for a few ms, after which
    # the first ~40 ms of work run up to 35 % slower (measured: 20-step repeats of 4.0, 3.5, 3.4, 3.1, 2.9, 2.9 ...
    # ms, identical from run to run): keep the device busy for >= 150 ms, then the W warm-up steps, right before the
    # timed repeats.  A count of steps, not a time, so that the timed steps compute the same thing on every run.
    for _ in range(BUSY_STEPS + args.warmup):
        dev_step()
    # The step time of this workload drifts by up to +-20 % over a few hundred steps (it follows the longest TOI chain /
    # largest island among the batch, and wedged agents stay wedged for a while): identical from run to run -- the
    # roll-out is deterministic -- but one short window lands in a slow or a fast stretch.  So the K timed steps are cut
    # into repeats spread over SPAN_STEPS steps of the roll-out, with untimed steps between them.
    sizes = repeat_sizes(args.steps, args.repeats)
    gap = math.ceil(max(0, SPAN_STEPS - args.steps) / (len(sizes) - 1)) if len(sizes) > 1 else 0
    reps, timed_launches = [], 0
    torch.cuda.profiler.start()        # `ncu --profile-from-start off` captures the timed repeats and the steps between them
    for i, n in enumerate(sizes):
        for _ in range(gap if i else 0):
            dev_step()
        l0 = sum(e_.kernel_launches() for e_ in envs)
        reps.append(timed(dev_step, n))
        timed_launches += sum(e_.kernel_launches() for e_ in envs) - l0
    torch.cuda.profiler.stop()
    dumped = None
    if args.dump_outputs and rank == 0:
        # what the last timed step returned, copied on the device before the arms below step the batches again
        last = envs[(tick[0] - 1) % ROT]._h
        names = list(env.obs_shapes()) + ['rewards', 'dones', 'episode_return', 'episode_length']
        outs = {k: last.tensor(k) for k in names + [k for k in ('immune', 'br_over', 'br_results') if last.has_tensor(k)]}
        idx = dump_sample(N, 4 + sum(4 * t[0].numel() for t in outs.values()), 1 + len(outs))
        sel = torch.as_tensor(idx, device=dev)
        dumped = {'env_index': idx, **{k: t.index_select(0, sel).to(torch.float32) for k, t in outs.items()}}
    clocks = clk.stop()
    ms_per_step = float(np.median([ms / n for ms, n in zip(reps, sizes)]))
    value = n_gpus * N * A / (ms_per_step * 1e-3)
    R = min(2000, max(args.repeats, math.ceil(SPAN_STEPS / args.steps)))    # repeats of K steps of the arms below

    # ---- the same loop with CUDA events around every kernel (roofline numerator) ---------------
    for e_ in envs:
        e_._h.kernel_timing(True)
    reps_k = [timed(dev_step, args.steps) for _ in range(max(5, min(R, 50)))]
    ksum, kn = np.zeros(3), 0
    for e_ in envs:
        ms3, n = e_._h.kernel_timing(False)
        ksum += np.array(ms3) * n; kn += n
    k_ms = ksum / max(kn, 1)                                   # mean ms of k_step, k_obs, k_lidar
    ms_per_step_kt = float(np.median(reps_k)) / args.steps
    stats = [e_.flush_stats() for e_ in envs]
    tot_steps = sum(s['steps'] for s in stats); tot_eps = sum(s['episodes'] for s in stats)

    # ---- end-to-end arms: host buffers through the C ABI ---------------------------------------
    def e2e_sync():      # H2D actions + kernels + D2H rewards/dones, host blocks until they arrived
        t = tick[0]; tick[0] += 1
        envs[t % ROT].step_host_async(acts_host[abatch(t)], rew_host[t % ROT], done_host[t % ROT])
        envs[t % ROT].step_host_wait()

    def e2e_pipelined():  # the same per-step copies, the ROT env groups in flight: a trainer that drives several env
        t = tick[0]; tick[0] += 1   # groups collects group r's rewards/dones while the other groups' steps run
        envs[t % ROT].step_host_wait()
        envs[t % ROT].step_host_async(acts_host[abatch(t)], rew_host[t % ROT], done_host[t % ROT])

    for _ in range(max(3, args.warmup)):
        e2e_sync()
    Re = int(max(5, min(R, 200)))
    e2e_sync_ms = float(np.median([timed(e2e_sync, args.steps) for _ in range(Re)])) / args.steps
    for _ in range(max(3, args.warmup)):
        e2e_pipelined()
    e2e_reps = [timed(e2e_pipelined, args.steps) for _ in range(Re)]
    e2e_ms = float(np.median(e2e_reps)) / args.steps
    for e_ in envs:
        e_.step_host_wait()
    e2e_value = n_gpus * N * A / (e2e_ms * 1e-3)
    checksum = float(sum(float(r.sum()) for r in rew_host))

    # ---- the ROT env groups each on a stream of their own (reported beside the headline, never instead of it) ----
    # `value` and `e2e` above step ONE 16 384-env group at a time through one stream, so every step waits for its
    # slowest block while most SMs idle.  A trainer that drives several env groups (the usual way to hide policy
    # inference) gives each group its own stream: the groups' steps then overlap and the tail of one is filled by
    # the next.  Same kernels, same per-step copies; only the scheduling differs.
    gstreams = [torch.cuda.Stream() for _ in range(ROT)]

    def timed_groups(fn, k, drain):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        cur = torch.cuda.current_stream()
        t0.record()
        for s_ in gstreams:
            s_.wait_stream(cur)
        for _ in range(k):
            fn()
        drain()
        for s_ in gstreams:
            cur.wait_stream(s_)
        t1.record()
        barrier()
        return max_over_ranks(float(t0.elapsed_time(t1)))

    def dev_step_groups():
        t = tick[0]; tick[0] += 1
        envs[t % ROT]._h.step(acts_dev[abatch(t)].data_ptr(), gstreams[t % ROT].cuda_stream)

    def e2e_groups():
        t = tick[0]; tick[0] += 1
        envs[t % ROT].step_host_wait()
        with torch.cuda.stream(gstreams[t % ROT]):
            envs[t % ROT].step_host_async(acts_host[abatch(t)], rew_host[t % ROT], done_host[t % ROT])

    def drain_hosts():       # inside the timed region: every group's rewards/dones have landed
        for e_ in envs:
            e_.step_host_wait()

    kg = max(args.steps, 3 * ROT)
    for _ in range(max(3, args.warmup) * ROT):
        dev_step_groups()
    torch.cuda.synchronize()
    grp_ms = float(np.median([timed_groups(dev_step_groups, kg, lambda: None) for _ in range(Re)])) / kg
    for _ in range(max(3, args.warmup) * ROT):
        e2e_groups()
    drain_hosts()
    grp_e2e_ms = float(np.median([timed_groups(e2e_groups, kg, drain_hosts) for _ in range(Re)])) / kg
    torch.cuda.synchronize()

    obs_bufs = [envs[r].host_obs_buffer() for r in range(ROT)]
    obs_bytes_host = envs[0]._h.obs_host_bytes()

    def e2e_obs_sync():  # ... + D2H of every observation tensor, one env group at a time
        t = tick[0]; tick[0] += 1
        envs[t % ROT].step_host_obs(acts_host[abatch(t)], obs_bufs[t % ROT][0], rew_host[t % ROT], done_host[t % ROT])

    def e2e_obs_pipelined():  # the ROT env groups in flight: group r's copy-out overlaps group r+1's kernels
        t = tick[0]; tick[0] += 1
        envs[t % ROT].step_host_wait()      # results of this group's previous step (the policy would read them here)
        envs[t % ROT].step_host_async(acts_host[abatch(t)], rew_host[t % ROT], done_host[t % ROT], obs_bufs[t % ROT][0])

    for _ in range(max(3, args.warmup)):
        e2e_obs_sync()
    Ro = int(max(5, min(R, 50)))
    e2e_obs_ms = float(np.median([timed(e2e_obs_sync, args.steps) for _ in range(Ro)])) / args.steps
    for _ in range(max(3, args.warmup)):
        e2e_obs_pipelined()
    e2e_pipe_ms = float(np.median([timed(e2e_obs_pipelined, args.steps) for _ in range(Ro)])) / args.steps
    for e_ in envs:
        e_.step_host_wait()
    obs_checksum = float(obs_bufs[0][1]['agent'][:, :, -6:].astype(np.float64).sum())

    bytes_env = env.bytes_per_env_step()            # whole step (k_step + k_obs2 [+ k_lidar])
    kstep_bytes = env._h.kernel_bytes_per_env(0)    # k_step: state read + written, actions, rewards, dones, camera words
    kbytes = [env._h.kernel_bytes_per_env(w) for w in range(3)]
    peak, peak_src = measured_peak()
    kavg_ms = float(k_ms[0])
    achieved = kstep_bytes * N / (kavg_ms * 1e-3) / 1e9
    ctr = ncu_counters(args.workload)
    sm_hz = (clocks.get('sm_mhz') or 1965.0) * 1e6
    issue = None
    if ctr.get('warp_inst_per_launch') and ctr.get('envs_per_launch'):
        winst = ctr['warp_inst_per_launch'] * N / ctr['envs_per_launch']
        issue = {'bound': 'issue', 'warp_inst_per_launch': winst, 'issue_slots_per_clk': 148 * 4, 'sm_hz': sm_hz,
                 'min_ms_at_full_issue': winst / (148 * 4 * sm_hz) * 1e3,
                 'frac': winst / (148 * 4 * sm_hz) * 1e3 / kavg_ms, 'source': ctr.get('source')}
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': n_gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': config_block(args.workload, n_gpus, N),
        'tile_plan': env._h.tile_plan(),
        'l2': f'{ROT} batches of {N} envs stepped round-robin ({ROT} x {batch_bytes / 1e6:.0f} MB of state+outputs '
              f'{">" if ROT * batch_bytes > L2_BYTES else "<="} 126 MB L2): inputs larger than L2, no flush',
        'timing': {'method': 'K timed steps in repeats spread over the roll-out; each repeat: barrier+sync, CUDA events, max over '
                             'ranks; median of the repeats\' ms per step',
                   'repeats': len(sizes), 'repeat_steps': sizes, 'untimed_steps_between_repeats': gap, 'timed_ms_total': float(np.sum(reps)),
                   'rep_ms_min': float(np.min(reps)), 'rep_ms_max': float(np.max(reps)),
                   'rep_ms': [round(float(x), 4) for x in reps[:64]],
                   'preroll_steps_per_batch': args.preroll, 'rotating_batches': ROT,
                   'mean_episode_steps_in_timed_region': (tot_steps / tot_eps) if tot_eps else None,
                   'episodes_finished_in_timed_region': int(tot_eps),
                   'ms_per_step_with_kernel_events': ms_per_step_kt},
        'ms_per_step_by_episode_phase': phase_ms,
        'env_steps_per_sec': value / A,
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': N * A * 6, 'd2h_bytes_per_step': N * A * 4 + N,
                'ms_per_step': e2e_ms, 'repeats': Re, 'rep_ms': [round(float(x), 4) for x in e2e_reps[:32]],
                'api': f'MaSurvivalVec.step_host_async / step_host_wait -> msv_step_host_async/_wait, pinned host buffers: every step copies its '
                       f'actions in and its rewards/dones out; the {ROT} env groups are kept in flight (the host waits for a group\'s results right '
                       'before submitting that group\'s next step)',
                'sync': {'value': n_gpus * N * A / (e2e_sync_ms * 1e-3), 'ms_per_step': e2e_sync_ms,
                         'how': 'one group at a time: submit, then block until its rewards/dones are in host memory'},
                'reward_checksum': checksum},
        'e2e_obs': {'value': n_gpus * N * A / (e2e_obs_ms * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': N * A * 6,
                    'd2h_bytes_per_step': N * A * 4 + N + obs_bytes_host, 'ms_per_step': e2e_obs_ms,
                    'd2h_gbs': (N * A * 4 + N + obs_bytes_host) / (e2e_obs_ms * 1e-3) / 1e9,
                    'api': 'MaSurvivalVec.step_host_obs -> msv_step_host_obs: rewards, dones AND every observation tensor land in pinned host memory',
                    'pipelined': {'value': n_gpus * N * A / (e2e_pipe_ms * 1e-3), 'ms_per_step': e2e_pipe_ms,
                                  'how': f'{ROT} env groups in flight (msv_step_host_async/_wait): copy-out of one group overlaps the kernels of the next'},
                    'obs_checksum': obs_checksum},
        'concurrent_groups': {'value': n_gpus * N * A / (grp_ms * 1e-3), 'unit': UNIT, 'ms_per_step': grp_ms,
                              'e2e': {'value': n_gpus * N * A / (grp_e2e_ms * 1e-3), 'ms_per_step': grp_e2e_ms,
                                      'h2d_bytes_per_step': N * A * 6, 'd2h_bytes_per_step': N * A * 4 + N},
                              'how': f'NOT the headline: the same {ROT} env groups of {N} envs, each driven through a CUDA stream of its own '
                                     '(device-resident: msv_step; e2e: step_host_async/_wait with pinned host buffers, the last results '
                                     'awaited inside the timed region), so the groups\' steps overlap and one group\'s slowest blocks no '
                                     'longer idle the other SMs'},
        'gpu_launches': int(timed_launches),
        'clocks': clocks,
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': ctr.get('dram_bytes_per_launch'), 'kernel': W['kernel'], 'kernel_ms': kavg_ms,
                     'kernel_ms_all': {'k_step': float(k_ms[0]), 'k_obs': float(k_ms[1]), 'k_lidar': float(k_ms[2])},
                     'kernel_share_of_step': float(k_ms[0] / max(k_ms.sum(), 1e-9)),
                     'kernel_gbs_all': {n: (kbytes[j] * N / (k_ms[j] * 1e-3) / 1e9 if k_ms[j] > 0.004 else None) for j, n in enumerate(('k_step', 'k_obs', 'k_lidar'))},
                     'algorithmic_bytes_per_env_step_all': dict(zip(('k_step', 'k_obs', 'k_lidar'), kbytes)),
                     'algorithmic_bytes_per_env_step': kstep_bytes, 'whole_step_bytes_per_env_step': bytes_env,
                     'whole_step_gbs': bytes_env * N / (ms_per_step * 1e-3) / 1e9, 'peak_source': peak_src,
                     'issue': issue,
                     'note': 'latency/issue bound, not bandwidth bound: see DESIGN.md section 8'},
    }
    if rank == 0:
        if world == 1 and not args.no_cpu:
            line['cpu_baseline'] = cpu_baseline(args.workload, sample_envs=min(N, 4096), steps=300, preroll=min(args.preroll, 600))
            rp = ref_python_baseline(args.workload)
            if rp:
                line['cpu_baseline_ref_python'] = rp
            c1 = {k: ref_python_baseline(k) for k in ('1v1_default', '2v2')}     # BASELINE.json configs[0]: 1 env, 1000 steps, demo.py loop
            if all(c1.values()):
                line['cpu_baseline_config1'] = c1
        if dumped is not None:
            write_dump(args.dump_outputs, {k: v if isinstance(v, np.ndarray) else v.cpu().numpy() for k, v in dumped.items()})
        print(json.dumps(line))
    for e_ in envs:
        e_.close()
    if world > 1:
        dist.destroy_process_group()


def _cpu_batch(name, seed, sample_envs, threads):
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import pyoracle as po
    rec = workload_config(name, auto_reset=True)
    A = int(rec['n_agents'])
    b = po.OracleBatch(rec, seed, sample_envs, threads)
    b.reset()
    rng = np.random.default_rng(0)
    acts = np.zeros((NB_CPU, sample_envs, A, 6), dtype=np.uint8)
    acts[..., 0:3] = rng.integers(0, 3, size=(NB_CPU, sample_envs, A, 3))
    acts[..., 3:6] = rng.integers(0, 2, size=(NB_CPU, sample_envs, A, 3))
    return b, acts, A


def cpu_baseline(name, sample_envs, steps, preroll, threads=None):
    """The oracle port (reference semantics restated in C, oracle/) timed on this box's host
    cores on a bounded sample of the same stationary workload."""
    threads = threads or os.cpu_count() or 1
    b, acts, A = _cpu_batch(name, 1, sample_envs, threads)
    for t in range(preroll):
        b.step(acts[(t * 7) % NB_CPU])
    t0 = time.perf_counter()
    for t in range(steps):
        b.step(acts[(t * 7) % NB_CPU])
    dt = time.perf_counter() - t0
    b.close()
    return {'value': sample_envs * steps * A / dt, 'unit': UNIT, 'cores': threads, 'kind': 'port',
            'sample': f'{sample_envs} envs x {steps} steps of the {name} workload after a {preroll}-step pre-roll, {threads} host threads, C oracle (oracle/masurv_oracle.c)',
            'seconds': dt}


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    W = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    n_gpus = int(os.environ.get('WORLD_SIZE', args.gpus))
    N = args.envs or W['envs']
    # bounded sample of the workload: at most 4096 envs per "step" keeps pre-roll + K steps within minutes
    sample = min(N, 4096)
    b, acts, A = _cpu_batch(args.workload, args.seed, sample, threads)
    preroll = min(args.preroll, 1500)
    for t in range(preroll):                      # the same stationary episode mix as the GPU arm
        b.step(acts[(t * 7) % NB_CPU])
    for t in range(args.warmup):
        b.step(acts[(t * 7) % NB_CPU])
    reps, t = [], 0                               # seconds per step of each repeat of the K timed steps
    for n in repeat_sizes(args.steps, max(args.repeats, 5)):
        t0 = time.perf_counter()
        for _ in range(n):
            rewards, dones = b.step(acts[(t * 7) % NB_CPU])
            t += 1
        reps.append((time.perf_counter() - t0) / n)
    if args.dump_outputs:
        write_dump(args.dump_outputs, {'env_index': np.arange(sample), 'rewards': rewards, 'dones': dones})
    b.close()
    dt = float(np.median(reps)) * args.steps
    value = sample * args.steps * A / dt
    cb = {'value': value, 'unit': UNIT, 'cores': threads, 'kind': 'port',
          'sample': f'{sample} envs per step (bounded sample of the {N}-env workload), {preroll}-step pre-roll, median of {len(reps)} repeats, '
                    f'{threads} host threads, C oracle port; the reference\'s own pybox2d stack is not installable in this image'}
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': n_gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': config_block(args.workload, n_gpus, N),
        'sample_envs_per_step': sample,
        'cpu_baseline': cb,
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    rp = ref_python_baseline(args.workload)
    if rp:
        line['cpu_baseline_ref_python'] = rp
    print(json.dumps(line))


def main():
    sys.dont_write_bytecode = True    # the benchmark may run from a read-only tree: it writes nothing there
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='2v2', choices=sorted(WORKLOADS))
    ap.add_argument('--envs', type=int, default=0, help='environments per GPU (default: the workload\'s BASELINE count)')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--preroll', type=int, default=1500, help='untimed steps per batch before the timed region (stationary episode mix)')
    ap.add_argument('--repeats', type=int, default=15, help='at most this many repeats of >= 20 of the K timed steps (median reported; the step time drifts by a few % over hundreds of steps as wedged agents come and go, so the median wants more than a handful)')
    ap.add_argument('--rotate', type=int, default=0, help='independent env batches stepped round-robin (0: the workload\'s count, scaled to --envs; enough to exceed L2)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-phase', action='store_true', help='skip the per-episode-phase timing')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step returned to DIR/<name>.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_ours(args)


if __name__ == '__main__':
    main()
