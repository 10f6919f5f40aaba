#!/usr/bin/env python
"""What anti-aliased frames cost on the GPU now that the render kernel streams the canvas through the
Lanczos resize in chunks of rows (moog_render_dev.cuh render_env_aa).

    python scripts/aa_render_cost.py [--parent DIR] [--launches 30] [--rounds 2] [--bench-runs 5] [--parts 1,2,3]

Prints, with the card's name and power limit:
  1. the render kernel alone (moog_render of 4096 falling_balls20 envs, CUDA events, L2 overwritten
     before every launch): with --parent (a built checkout of the commit before), parent and this tree
     alternated at the sizes both can draw (64x64 at anti_aliasing 1, 2, 3); this tree alone at
     84x84 AA 3, 128x128 AA 2, 256x256 AA 2, 64x64 AA 4, and 256x256 AA 1 (the same canvas unaliased);
  2. step + frames of 4096 falling_balls20 envs with a 128x128 AA 2 view 0 (drawn by the render tail
     behind the step), next to 64x64 AA 1;
  3. with --parent: bench.py of the parent and of this tree, alternated, --bench-runs each.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = 'power limit not readable'
    return '{} ({})'.format(name, q)


# run inside a given tree: falling_balls20 x 4096 envs with view 0 = PILRenderer(image_size=(w, h),
# anti_aliasing=aa), stepped 20 times; then either the render kernel alone or step + frames
_RUN = r'''
import sys, importlib, numpy as np, torch
tree, what, w, h, aa, launches = sys.argv[1], sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5]), int(sys.argv[6])
sys.path.insert(0, tree)
import moog_b200
from moog import observers
from moog_b200.batched_env import BatchedEnvironment
cfg = importlib.import_module('moog_b200.configs.falling_balls20').get_config()
cfg['observers'] = {'image': observers.PILRenderer(image_size=(w, h), anti_aliasing=aa)}
np.random.seed(1234)
states = [cfg['state_initializer']() for _ in range(512)]
N = 4096
env = BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=1234, initial_states=states)
env.reset()
eng = env.engine
act = torch.from_numpy(np.random.RandomState(1).randint(0, 5, size=(N, 1)).astype(np.float64)).cuda()
for _ in range(20):
    eng.env_step(act, frames=True)
flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda:0')
call = (lambda: eng.render()) if what == 'render' else (lambda: eng.env_step(act, frames=True))
for _ in range(5):
    call()
ev = []
for _ in range(launches):
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); call(); b.record()
    ev.append((a, b))
torch.cuda.synchronize()
us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
print('US', np.median(us), us.min(), us.max())
'''


def _run(tree, what, w, h, aa, launches):
    out = subprocess.run([sys.executable, '-c', _RUN, tree, what, str(w), str(h), str(aa), str(launches)],
                         capture_output=True, text=True, cwd=tree)
    for line in out.stdout.splitlines():
        if line.startswith('US '):
            return [float(v) for v in line.split()[1:]]
    raise RuntimeError('{} {}x{} aa{} in {} failed:\n{}'.format(what, w, h, aa, tree, out.stderr[-3000:]))


def _bench(tree):
    out = subprocess.run([sys.executable, 'bench.py', '--gpus', '1', '--no-cpu'], capture_output=True, text=True,
                         cwd=tree)
    for line in out.stdout.splitlines()[::-1]:
        if line.startswith('{'):
            return json.loads(line)['value']
    raise RuntimeError('bench.py in {} failed:\n{}'.format(tree, out.stderr[-3000:]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--parent', default=None, help='a built checkout of the commit before this change')
    ap.add_argument('--launches', type=int, default=30)
    ap.add_argument('--rounds', type=int, default=2)
    ap.add_argument('--bench-runs', type=int, default=5)
    ap.add_argument('--parts', default='1,2,3', help='which of the numbered measurements to run')
    args = ap.parse_args()
    parts = {int(p) for p in args.parts.split(',')}
    print('card:', _card())
    fmt = lambda r: 'median %.1f us (min %.1f, max %.1f)' % tuple(r)
    if 1 in parts:
        _part1(args, fmt)
    if 2 in parts:
        print('2. step + frames (env_step, frames=True), 4096 falling_balls20 envs, view 0 drawn behind the step')
        for w, h, aa in [(64, 64, 1), (128, 128, 2)]:
            print('  %3dx%-3d AA %d: %s' % (w, h, aa, fmt(_run(ROOT, 'step', w, h, aa, args.launches))))
            sys.stdout.flush()
    if 3 in parts and args.parent:
        _part3(args)
    print('card:', _card())


def _part1(args, fmt):
    print('1. moog_render, 4096 falling_balls20 frames, %d launches per run, L2 overwritten before each' % args.launches)
    shared = [(64, 64, 1), (64, 64, 2), (64, 64, 3)]
    for w, h, aa in shared:
        for rnd in range(args.rounds):
            trees = ([('parent', args.parent)] if args.parent else []) + [('this tree', ROOT)]
            for name, tree in trees:
                print('  %3dx%-3d AA %d  %-9s round %d: %s' % (w, h, aa, name, rnd, fmt(_run(tree, 'render', w, h, aa,
                                                                                               args.launches))))
                sys.stdout.flush()
    for w, h, aa in [(84, 84, 3), (128, 128, 2), (256, 256, 2), (64, 64, 4), (256, 256, 1)]:
        print('  %3dx%-3d AA %d  this tree        : %s' % (w, h, aa, fmt(_run(ROOT, 'render', w, h, aa, args.launches))))
        sys.stdout.flush()


def _part3(args):
    print('3. bench.py (falling_balls20, 4096 envs, 64x64 AA 1), alternated, %d runs each' % args.bench_runs)
    vals = {'parent': [], 'this tree': []}
    for _ in range(args.bench_runs):
        for name, tree in (('parent', args.parent), ('this tree', ROOT)):
            vals[name].append(_bench(tree))
            print('  %-9s run %d: %.0f env-steps/s' % (name, len(vals[name]), vals[name][-1]))
            sys.stdout.flush()
    for name, v in vals.items():
        print('  %-9s: median %.0f env-steps/s (min %.0f, max %.0f) runs %s' % (
            name, np.median(v), min(v), max(v), ', '.join('%.0f' % x for x in v)))
    print('  this tree / parent (medians) = %.4f' % (np.median(vals['this tree']) / np.median(vals['parent'])))


if __name__ == '__main__':
    main()
