#!/usr/bin/env python
"""What SpriteMask observers (moog_render_mask) cost on the GPU, and that a program without one costs what it did.

    python scripts/mask_cost.py [--parent DIR] [--bench-rounds 3] [--steps 40] [--rounds 4] [--out FILE]

Writes (to --out, default profiles/r08_mask_cost.txt, and to stdout), with the card's name and power limit:
  1. the mask kernel alone next to the RGB render kernel, per 4096 falling_balls20 envs at 64 x 64 and
     256 x 256 (CUDA events, every shape warmed up, L2 overwritten before each launch), and the kernels'
     `-Xptxas -v` registers and spills;
  2. falling_balls20 at 4096 envs, device-resident: step + frames without a mask and with a 64 x 64 mask,
     the arms alternated in `--rounds` windows of `--steps`;
  3. HostPipeline(depth=2) end to end with a 64 x 64 mask, 'mapped' and 'device', next to no mask;
  4. with --parent (a built checkout of the parent commit): bench.py of the parent and of this tree,
     alternated in the same run.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

_LINES = []


def say(text):
    print(text, flush=True)
    _LINES.append(text)


def _card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'power limit not readable'
    return '{} ({})'.format(name, q)


def _ptxas():
    """`-Xptxas -v` registers and spills of the render and mask kernels of this tree."""
    import tempfile
    from moog_b200 import build
    src = os.path.join(ROOT, 'moog.github.io_b200', 'csrc', 'moog_render.cu')
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [build._nvcc()] + build.NVCC_FLAGS + ['-Xptxas', '-v', '-c', src, '-o', os.path.join(tmp, 'r.o')]
        out = subprocess.run(cmd, capture_output=True, text=True).stderr
    res, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Compiling entry function '_ZN4moog\d+(\w+?)E", line)
        if m:
            cur = m.group(1)
        m = re.search(r'(\d+) bytes spill stores, (\d+) bytes spill loads', line)
        if m and cur:
            res.setdefault(cur, {})['spills'] = '{} B st / {} B ld'.format(*m.groups())
        m = re.search(r'Used (\d+) registers', line)
        if m and cur:
            res.setdefault(cur, {})['regs'] = int(m.group(1))
    return res


def _env(n, extra=None, pool=512, seed=1234):
    import moog_b200  # noqa: F401
    import importlib
    from moog_b200.batched_env import BatchedEnvironment
    cfg = importlib.import_module('moog_b200.configs.falling_balls20').get_config()
    if extra:
        cfg['observers'] = dict(cfg['observers'], **extra)
    np.random.seed(seed)
    states = [cfg['state_initializer']() for _ in range(pool)]
    return BatchedEnvironment(**cfg, num_envs=n, device='cuda:0', seed=seed, initial_states=states)


def _mask(size):
    from moog import observers
    return observers.SpriteMask(image_size=(size, size))


def _renderer(size):
    from moog import observers
    return observers.PILRenderer(image_size=(size, size))


def _actions(n, seed=1):
    import torch
    rng = np.random.RandomState(seed)
    return torch.from_numpy(rng.randint(0, 5, size=(n, 1)).astype(np.float64)).to('cuda:0')


def _burn_in(env, actions, steps=130, episode=100):
    """bench.py's burn-in: every env reset once at a random step, so the batch holds a mix of phases."""
    import torch
    eng = env.engine
    env.reset()
    phase = torch.randint(0, episode, (env.num_envs,), generator=torch.Generator().manual_seed(0)).to(eng.device)
    for t in range(steps):
        if t < episode:
            eng.state.envi[:, 1] = torch.where(phase == t, torch.ones_like(eng.state.envi[:, 1]), eng.state.envi[:, 1])
        eng.env_step(actions, frames=True)
    torch.cuda.synchronize()


def kernels(launches):
    import torch
    for k, v in sorted(_ptxas().items()):
        say('  ptxas {:<40}: {} registers, spills {}'.format(k, v.get('regs'), v.get('spills')))
    n = 4096
    env = _env(n, dict(v256=_renderer(256), m64=_mask(64), m256=_mask(256)))
    _burn_in(env, _actions(n))
    eng = env.engine
    arms = [('moog_render_kernel, 64x64 frames', lambda: eng.render(view=0)),
            ('moog_render_mask_kernel, 64x64 masks', lambda: eng.render_mask(mask=0)),
            ('moog_render_kernel, 256x256 frames', lambda: eng.render(view=1)),
            ('moog_render_mask_kernel, 256x256 masks', lambda: eng.render_mask(mask=1))]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda:0')
    for _, fn in arms:          # every shape warmed up
        for _ in range(5):
            fn()
    times = {label: [] for label, _ in arms}
    for _ in range(launches):
        for label, fn in arms:
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            times[label].append((a, b))
    torch.cuda.synchronize()
    for label, ev in times.items():
        us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
        say('  {:<40}: median {:.1f} us per 4096 envs (min {:.1f}, max {:.1f}; {} launches, L2 overwritten '
            'before each)'.format(label, np.median(us), us.min(), us.max(), launches))
    del env, eng
    torch.cuda.empty_cache()


def step_with_mask(steps, rounds):
    import torch
    n = 4096
    arms = {'no mask': _env(n), '+ 64x64 mask': _env(n, dict(mask=_mask(64)))}
    act = _actions(n)
    for env in arms.values():
        _burn_in(env, act)
    res = {k: [] for k in arms}
    for r in range(rounds + 1):                       # round 0 warms up
        for label, env in arms.items():
            eng = env.engine
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                eng.env_step(act, frames=True)
                for m in range(len(eng.masks)):
                    eng.render_mask(mask=m)
            b.record()
            b.synchronize()
            if r:
                res[label].append(a.elapsed_time(b) / steps)
    base = np.median(res['no mask'])
    for label, v in res.items():
        say('  {:<14}: {:.3f} ms / step median of {} windows x {} steps (min {:.3f}, max {:.3f}); {:+.3f} ms '
            '= {:+.1f} % vs no mask'.format(label, np.median(v), rounds, steps, min(v), max(v),
                                           np.median(v) - base, 100 * (np.median(v) - base) / base))
    del arms
    torch.cuda.empty_cache()


def pipeline_rate(steps, rounds):
    import torch
    n = 4096
    act = _actions(n)
    for extra in (None, dict(mask=_mask(64))):
        env = _env(n, extra)
        _burn_in(env, act, steps=60, episode=60)
        for mode in ('mapped', 'device'):
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
            label = '{}, {}'.format('64x64 frames + 64x64 mask' if extra else '64x64 frames only', mode)
            say('  {:<34}: {:.3f} M env-steps/s median of {} windows x {} steps (min {:.3f}, max {:.3f})'.format(
                label, np.median(rates) / 1e6, rounds, steps, min(rates) / 1e6, max(rates) / 1e6))
        del env
        torch.cuda.empty_cache()


def bench_ab(parent, rounds):
    trees = (('parent', parent), ('this tree', ROOT))
    bench = {t: [] for t, _ in trees}
    for r in range(rounds):
        for label, tree in (trees if r % 2 == 0 else trees[::-1]):
            out = subprocess.run([sys.executable, 'bench.py', '--gpus', '1', '--steps', '20', '--warmup', '3'],
                                 cwd=tree, capture_output=True, text=True)
            line = [l for l in out.stdout.splitlines() if l.startswith('{')]
            if out.returncode != 0 or not line:
                raise SystemExit('bench.py failed in {}: {}'.format(tree, out.stderr[-2000:]))
            res = json.loads(line[-1])
            bench[label].append((res['value'], res['ms_per_step']))
    for label, _ in trees:
        v = np.array(bench[label])
        say('  bench.py {:<9}: {:.0f} env-steps/s median of {} runs (min {:.0f}, max {:.0f}); ms_per_step {}'.format(
            label, np.median(v[:, 0]), len(v), v[:, 0].min(), v[:, 0].max(), ', '.join('{:.3f}'.format(x) for x in v[:, 1])))
    p, b = np.median(np.array(bench['parent'])[:, 0]), np.median(np.array(bench['this tree'])[:, 0])
    say('  headline this tree / parent = {:.4f}'.format(b / p))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--parent', help='built checkout of the parent commit for the same-run bench.py A/B')
    ap.add_argument('--bench-rounds', type=int, default=3)
    ap.add_argument('--launches', type=int, default=100)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=4)
    ap.add_argument('--bench-only', action='store_true', help='only section 4 (with --parent)')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r08_mask_cost.txt'))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('mask_cost.py needs a CUDA device')
    say('card: {}'.format(_card()))
    if not args.bench_only:
        say('1. kernels alone, falling_balls20 x 4096 envs')
        kernels(args.launches)
        say('2. falling_balls20 x 4096 envs, device-resident: step + frames, the mask drawn behind the step')
        step_with_mask(args.steps, args.rounds)
        say('3. HostPipeline(depth=2), falling_balls20 x 4096 envs, end to end (host clock, pinned TimeSteps '
            'collected)')
        pipeline_rate(max(args.steps // 2, 10), args.rounds)
    if args.parent:
        say('4. bench.py (4096 falling_balls20 envs, no mask): parent vs this tree, alternated in this run')
        bench_ab(os.path.abspath(args.parent), args.bench_rounds)
    say('card: {}'.format(_card()))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write('\n'.join(_LINES) + '\n')


if __name__ == '__main__':
    main()
