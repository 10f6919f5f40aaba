#!/usr/bin/env python
"""What further PILRenderer views (moog_render_view) cost on the GPU, and that one view costs what it did.

    python scripts/views_cost.py [--parent DIR] [--bench-rounds 3] [--steps 40] [--rounds 4]

Prints, with the card's name and power limit:
  1. with --parent (a built checkout of the commit before views existed): bench.py of the parent and of
     this tree, alternated in the same run, plus the render kernel's own time (CUDA events, L2
     overwritten between launches, 4096 falling_balls20 envs) and its `-Xptxas -v` registers and spills
     in each tree;
  2. falling_balls20 at 4096 envs, device-resident: step + frames with one view, and with a second
     view at 64 x 64 and at 128 x 128 into HBM, the arms alternated in `--rounds` windows of `--steps`;
  3. HostPipeline(depth=2) end to end with two views (64 x 64 + 128 x 128), 'mapped' vs 'device', next to
     one view.
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


def _card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'power limit not readable'
    return '{} ({})'.format(name, q)


# the render kernel alone, run inside a given tree: moog_render (view 0) of 4096 falling_balls20 envs
_RENDER_TIME = r'''
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1])
import moog_b200, importlib
from moog_b200.batched_env import BatchedEnvironment
cfg = importlib.import_module('moog_b200.configs.falling_balls20').get_config()
np.random.seed(1234)
states = [cfg['state_initializer']() for _ in range(512)]
env = BatchedEnvironment(**cfg, num_envs=4096, device='cuda:0', seed=1234, initial_states=states)
env.reset()
act = torch.from_numpy(np.random.RandomState(1).randint(0, 5, size=(4096, 1)).astype(np.float64)).cuda()
for _ in range(60):
    env.engine.env_step(act, frames=True)
eng = env.engine
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda:0')
for _ in range(5):
    eng.render()
ev = []
for _ in range(int(sys.argv[2])):
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); eng.render(); b.record()
    ev.append((a, b))
torch.cuda.synchronize()
us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
print('RENDER_US', np.median(us), us.min(), us.max())
'''


def _ptxas(tree):
    """`-Xptxas -v` lines of the render kernels of `tree` (compiled to a temporary object)."""
    import tempfile
    sys.path.insert(0, ROOT)
    from moog_b200 import build
    src = os.path.join(tree, 'moog.github.io_b200', 'csrc', 'moog_render.cu')
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [build._nvcc()] + build.NVCC_FLAGS + ['-Xptxas', '-v', '-c', src, '-o', os.path.join(tmp, 'r.o')]
        out = subprocess.run(cmd, capture_output=True, text=True).stderr
    res, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Compiling entry function '_ZN4moog\d+(\w+?)ENS", line)
        if m:
            cur = m.group(1)
        m = re.search(r'(\d+) bytes spill stores, (\d+) bytes spill loads', line)
        if m and cur:
            res.setdefault(cur, {})['spills'] = '{} B st / {} B ld'.format(*m.groups())
        m = re.search(r'Used (\d+) registers', line)
        if m and cur:
            res.setdefault(cur, {})['regs'] = int(m.group(1))
    return res


def ab(parent, rounds, launches):
    trees = (('parent', parent), ('this tree', ROOT))
    for label, tree in trees:
        for k, v in sorted(_ptxas(tree).items()):
            print('  ptxas {:<9} {:<36}: {} registers, spills {}'.format(label, k, v.get('regs'), v.get('spills')))
    bench, render = {t: [] for t, _ in trees}, {t: [] for t, _ in trees}
    for r in range(rounds):
        for label, tree in (trees if r % 2 == 0 else trees[::-1]):
            out = subprocess.run([sys.executable, 'bench.py', '--gpus', '1', '--steps', '20', '--warmup', '3'],
                                 cwd=tree, capture_output=True, text=True)
            line = [l for l in out.stdout.splitlines() if l.startswith('{')]
            if out.returncode != 0 or not line:
                raise SystemExit('bench.py failed in {}: {}'.format(tree, out.stderr[-2000:]))
            res = json.loads(line[-1])
            bench[label].append((res['value'], res['ms_per_step'],
                                 res['roofline']['render_kernel']['kernel_ms'] if 'render_kernel' in res.get(
                                     'roofline', {}) else float('nan')))
            out = subprocess.run([sys.executable, '-c', _RENDER_TIME, tree, str(launches)], capture_output=True,
                                 text=True)
            m = re.search(r'RENDER_US (\S+) (\S+) (\S+)', out.stdout)
            if not m:
                raise SystemExit('render timing failed in {}: {}'.format(tree, out.stderr[-2000:]))
            render[label].append(tuple(float(x) for x in m.groups()))
    for label, _ in trees:
        v = np.array(bench[label])
        print('  bench.py {:<9}: {:.0f} env-steps/s median of {} runs (min {:.0f}, max {:.0f}); ms_per_step {}; '
              'bench render kernel_ms {}'.format(label, np.median(v[:, 0]), len(v), v[:, 0].min(), v[:, 0].max(),
                                                 ', '.join('{:.3f}'.format(x) for x in v[:, 1]),
                                                 ', '.join('{:.3f}'.format(x) for x in v[:, 2])))
        rv = np.array(render[label])
        print('  moog_render_kernel {:<9}: median {} us per 4096 64x64 frames ({} launches per run, L2 '
              'overwritten before each; per run min {})'.format(label, ', '.join('{:.1f}'.format(x) for x in rv[:, 0]),
                                                               launches, ', '.join('{:.1f}'.format(x) for x in rv[:, 1])))
    p, b = np.median(np.array(bench['parent'])[:, 0]), np.median(np.array(bench['this tree'])[:, 0])
    print('  headline this tree / parent = {:.4f}'.format(b / p))


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


def _renderer(size):
    from moog import observers
    return observers.PILRenderer(image_size=(size, size), anti_aliasing=1)


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


def _actions(n, seed=1):
    import torch
    rng = np.random.RandomState(seed)
    return torch.from_numpy(rng.randint(0, 5, size=(n, 1)).astype(np.float64)).to('cuda:0')


def step_with_views(steps, rounds):
    import torch
    n = 4096
    arms = {'one view (64x64)': _env(n), '+ second view 64x64': _env(n, dict(v64=_renderer(64))),
            '+ second view 128x128': _env(n, dict(v128=_renderer(128)))}
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
                for v in range(1, eng.n_views):
                    eng.render(view=v)
            b.record()
            b.synchronize()
            if r:
                res[label].append(a.elapsed_time(b) / steps)
    base = np.median(res['one view (64x64)'])
    for label, v in res.items():
        print('  {:<22}: {:.3f} ms / step median of {} windows x {} steps (min {:.3f}, max {:.3f}); {:+.3f} ms '
              '= {:+.1f} % vs one view'.format(label, np.median(v), rounds, steps, min(v), max(v),
                                              np.median(v) - base, 100 * (np.median(v) - base) / base))
    del arms
    torch.cuda.empty_cache()


def pipeline_rate(steps, rounds):
    import torch
    n = 4096
    act = _actions(n)
    for extra, modes in ((None, ('mapped', 'device')), (dict(v128=_renderer(128)), ('mapped', 'device'))):
        env = _env(n, extra)
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
            label = '{}, {}'.format('64x64 + 128x128' if extra else '64x64 only', mode)
            print('  {:<24}: {:.3f} M env-steps/s median of {} windows x {} steps (min {:.3f}, max {:.3f})'.format(
                label, np.median(rates) / 1e6, rounds, steps, min(rates) / 1e6, max(rates) / 1e6))
        del env
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--parent', help='built checkout of the parent commit for the same-run A/B')
    ap.add_argument('--bench-rounds', type=int, default=3)
    ap.add_argument('--launches', type=int, default=200)
    ap.add_argument('--steps', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=4)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('views_cost.py needs a CUDA device')
    print('card: {}'.format(_card()))
    if args.parent:
        print('1. single-renderer regression check: parent vs this tree, alternated in this run')
        ab(os.path.abspath(args.parent), args.bench_rounds, args.launches)
    print('2. falling_balls20 x 4096 envs, device-resident: step + frames, further views drawn behind the step')
    step_with_views(args.steps, args.rounds)
    print('3. HostPipeline(depth=2), falling_balls20 x 4096 envs, end to end (host clock, pinned TimeSteps collected)')
    pipeline_rate(max(args.steps // 2, 10), args.rounds)
    print('card: {}'.format(_card()))


if __name__ == '__main__':
    main()
