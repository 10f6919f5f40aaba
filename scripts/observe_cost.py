#!/usr/bin/env python
"""What the RawState observation (moog_observe_sprites, csrc/moog_observe.cu) costs on the GPU.

    python scripts/observe_cost.py [--launches 200] [--steps 40] [--rounds 4]

Prints, with the card's name and power limit:
  1. the kernel's own time (CUDA events around every launch, L2 overwritten between launches) for
     falling_balls20 at 4096 envs and synthetic32 at 131 072 envs, into HBM and into pinned host memory,
     with the bytes it must move per env;
  2. falling_balls20 at 4096 envs, device-resident: step (frames included, as bench.py times it)
     against step + observation, the two alternated in `--rounds` windows of `--steps` steps;
  3. HostPipeline(depth=2) end to end, synthetic32 state only at 131 072 envs: without an observer,
     and with RawState over both transports ('mapped', 'device').
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'power limit not readable'
    return '{} ({})'.format(name, q)


def _env(scene, n, raw_state, state_only=False, pool=256, seed=1234):
    import moog_b200  # noqa: F401
    import importlib
    from moog import observers
    from moog_b200.batched_env import BatchedEnvironment
    cfg = importlib.import_module('moog_b200.configs.' + scene).get_config()
    obs = {} if state_only else dict(cfg['observers'])
    if raw_state:
        obs['state'] = observers.RawState()
    cfg['observers'] = obs
    np.random.seed(seed)
    states = [cfg['state_initializer']() for _ in range(pool)]
    return BatchedEnvironment(**cfg, num_envs=n, device='cuda:0', seed=seed, initial_states=states)


def _burn_in(env, actions, steps=130, episode=100):
    """bench.py's burn-in: every env reset once at a random step, so the batch holds a mix of phases."""
    import torch
    eng = env.engine
    env.reset()
    phase = torch.randint(0, episode, (env.num_envs,), generator=torch.Generator().manual_seed(0)).to(eng.device)
    for t in range(steps):
        if t < episode:
            eng.state.envi[:, 1] = torch.where(phase == t, torch.ones_like(eng.state.envi[:, 1]), eng.state.envi[:, 1])
        eng.env_step(actions, frames=True if eng.frames is not None else None)
    torch.cuda.synchronize()


def _grid_actions(env, seed=1):
    import torch
    rng = np.random.RandomState(seed)
    return torch.from_numpy(rng.randint(0, 5, size=(env.num_envs, env.action_dim)).astype(np.float64)).to('cuda:0')


def kernel_time(env, launches, label):
    import torch
    eng, prog = env.engine, env.program
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda:0')       # > 126 MB of L2
    host = torch.empty(eng.sprites.shape, dtype=torch.float32).pin_memory()
    cnt = eng.state.cnt.cpu().numpy()[:, :prog.n_layers]
    live = float(cnt.sum(axis=1).mean())
    # bytes the kernel moves per env: 13 float64 rows + 1 int32 row of every live slot, the env's counts,
    # 64 bytes per slot out
    rd = live * (13 * 8 + 4) + 4 * prog.n_layers
    wr = prog.n_slots * 64
    for where, out in (('HBM', eng.sprites), ('pinned host', host)):
        for _ in range(5):
            eng.observe_sprites(out=out)
        times = []
        for _ in range(launches):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.observe_sprites(out=out)
            b.record()
            times.append((a, b))
        torch.cuda.synchronize()
        us = np.array([a.elapsed_time(b) * 1e3 for a, b in times])
        print('  {:<34} -> {:<11}: median {:8.1f} us  (min {:.1f}, max {:.1f}, {} launches, L2 overwritten '
              'before each); {:.2f} KB read + {:.2f} KB written per env, {:.1f} MB + {:.1f} MB per call = '
              '{:.0f} GB/s'.format(label, where, np.median(us), us.min(), us.max(), launches, rd / 1e3, wr / 1e3,
                                   rd * env.num_envs / 1e6, wr * env.num_envs / 1e6,
                                   (rd + wr) * env.num_envs / (np.median(us) * 1e-6) / 1e9))
    del flush


def step_vs_observe(steps, rounds):
    import torch
    env = _env('falling_balls20', 4096, raw_state=True, pool=512)
    eng = env.engine
    act = _grid_actions(env)
    _burn_in(env, act)
    res = {'step': [], 'step + observation': []}
    for r in range(rounds + 1):                       # round 0 warms up
        for arm in res:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                eng.env_step(act, frames=True)
                if arm != 'step':
                    eng.observe_sprites()
            b.record()
            b.synchronize()
            if r:
                res[arm].append(a.elapsed_time(b) / steps)
    base = np.median(res['step'])
    for arm, v in res.items():
        print('  {:<20}: {:.3f} ms / step median of {} windows x {} steps (min {:.3f}, max {:.3f})'.format(
            arm, np.median(v), rounds, steps, min(v), max(v)))
    d = np.median(res['step + observation']) - base
    diffs = [b - a for a, b in zip(res['step'], res['step + observation'])]
    print('  observation adds {:+.3f} ms / step = {:+.2f} % of the step (per-window differences {})'.format(
        d, 100 * d / base, ', '.join('{:+.3f}'.format(x) for x in diffs)))


def pipeline_rate(steps, rounds):
    import torch
    n = 131072
    for raw_state, modes in ((False, ('mapped',)), (True, ('mapped', 'device'))):
        env = _env('synthetic32', n, raw_state=raw_state, state_only=True, pool=512)
        act = _grid_actions(env)
        _burn_in(env, act, steps=60, episode=60)
        for mode in modes:
            pipe = env.host_pipeline(depth=2, frames=mode)
            rates = []
            for r in range(rounds + 1):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                pipe.submit(act)
                for _ in range(steps - 1):
                    pipe.submit(act)
                    pipe.collect()
                pipe.collect()
                dt = time.perf_counter() - t0
                if r:
                    rates.append(steps * n / dt)
            label = 'RawState, {}'.format(mode) if raw_state else 'no observer'
            print('  {:<20}: {:.3f} M env-steps/s median of {} windows x {} steps (min {:.3f}, max {:.3f})'.format(
                label, np.median(rates) / 1e6, rounds, steps, min(rates) / 1e6, max(rates) / 1e6))
        del env
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--launches', type=int, default=200)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=4)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('observe_cost.py needs a CUDA device')
    print('card: {}'.format(_card()))
    print('1. moog_observe_kernel alone')
    for scene, n in (('falling_balls20', 4096), ('synthetic32', 131072)):
        env = _env(scene, n, raw_state=True, state_only=(scene == 'synthetic32'), pool=512)
        _burn_in(env, _grid_actions(env), steps=60, episode=60)
        kernel_time(env, args.launches, '{} x {} envs (S = {})'.format(scene, n, env.program.n_slots))
        del env
        torch.cuda.empty_cache()
    print('2. falling_balls20 x 4096 envs, device-resident, frames drawn by the step call')
    step_vs_observe(args.steps, args.rounds)
    print('3. HostPipeline(depth=2), synthetic32 state only x 131072 envs, end to end (host clock, pinned '
          'TimeSteps collected)')
    pipeline_rate(max(args.steps // 2, 10), args.rounds)


if __name__ == '__main__':
    main()
