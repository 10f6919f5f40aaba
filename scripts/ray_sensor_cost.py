#!/usr/bin/env python
"""What RaySensor observers (moog_ray_sensor) cost on the GPU, and that a program without one costs what it did.

    python scripts/ray_sensor_cost.py [--parent DIR] [--bench-rounds 3] [--steps 40] [--rounds 4] [--out FILE]

Writes (to --out, default profiles/r09_ray_sensor_cost.txt, and to stdout), with the card's name and power limit:
  1. the ray kernel alone at 32 and 256 rays next to the 64 x 64 SpriteMask kernel, per 4096 envs of
     colliding_predators84 (origin: the agent) and falling_balls20 (origin: ball 0; the scene's agent layer is
     empty), CUDA events, every shape warmed up, L2 overwritten before each launch; and the kernel's
     `-Xptxas -v` registers and spills;
  2. the same scenes at 4096 envs, device-resident: step + frames without a sensor and with one 32-ray sensor
     cast behind the step, the arms alternated in `--rounds` windows of `--steps`;
  3. with --parent (a built checkout of the parent commit): bench.py of the parent and of this tree,
     alternated in the same run.
"""
import argparse
import importlib
import json
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

_LINES = []

# scene -> (agent layer, agent index) of the sensors
SCENES = {'colliding_predators84': ('agent', 0), 'falling_balls20': ('balls', 0)}


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
    """`-Xptxas -v` registers, shared memory and spills of the ray kernel of this tree."""
    import tempfile
    from moog_b200 import build
    src = os.path.join(ROOT, 'moog.github.io_b200', 'csrc', 'moog_rays.cu')
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [build._nvcc()] + build.NVCC_FLAGS + ['-Xptxas', '-v', '-c', src, '-o', os.path.join(tmp, 'r.o')]
        out = subprocess.run(cmd, capture_output=True, text=True).stderr
    return [l.strip() for l in out.splitlines() if re.search(r'spill|Used \d+ registers', l)]


def _env(scene, n, extra=None, pool=512, seed=1234):
    import moog_b200  # noqa: F401
    from moog_b200.batched_env import BatchedEnvironment
    mod = importlib.import_module('moog_b200.configs.' + scene)
    cfg = mod.get_config()
    if extra:
        cfg['observers'] = dict(cfg['observers'], **extra)
    np.random.seed(seed)
    states = [cfg['state_initializer']() for _ in range(pool)]
    return BatchedEnvironment(**cfg, num_envs=n, device='cuda:0', seed=seed, initial_states=states,
                              layer_capacity=getattr(mod, 'LAYER_CAPACITY', None))


def _sensor(scene, rays):
    import moog_b200  # noqa: F401  (puts the package's `moog` on the path)
    from moog import observers
    layer, index = SCENES[scene]
    return observers.RaySensor(layer, num_rays=rays, agent_index=index)


def _actions(env, seed=1):
    import torch
    rng = np.random.RandomState(seed)
    if env.action_dim == 1:
        a = rng.randint(0, 5, size=(env.num_envs, 1)).astype(np.float64)
    else:
        a = rng.uniform(-1, 1, size=(env.num_envs, env.action_dim))
    return torch.from_numpy(a).to('cuda:0')


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
    import moog_b200  # noqa: F401
    from moog import observers
    for line in _ptxas():
        say('  ptxas: ' + line)
    n = 4096
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda:0')
    for scene in SCENES:
        env = _env(scene, n, dict(r32=_sensor(scene, 32), r256=_sensor(scene, 256),
                                  m64=observers.SpriteMask(image_size=(64, 64))))
        _burn_in(env, _actions(env))
        eng = env.engine
        hits = [float((eng.sense_rays(sensor=k)[..., 1] >= 0).float().mean()) for k in range(2)]
        arms = [('moog_ray_sensor_kernel, 32 rays', lambda: eng.sense_rays(sensor=0)),
                ('moog_ray_sensor_kernel, 256 rays', lambda: eng.sense_rays(sensor=1)),
                ('moog_render_mask_kernel, 64x64 masks', lambda: eng.render_mask(mask=0))]
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
        say('  {} x 4096 envs ({:.1f} % / {:.1f} % of the 32 / 256 rays meet a sprite):'.format(
            scene, 100 * hits[0], 100 * hits[1]))
        for label, ev in times.items():
            us = np.array([a.elapsed_time(b) * 1e3 for a, b in ev])
            say('    {:<38}: median {:.1f} us (min {:.1f}, max {:.1f}; {} launches, L2 overwritten before '
                'each)'.format(label, np.median(us), us.min(), us.max(), launches))
        del env, eng
        torch.cuda.empty_cache()


def step_with_sensor(steps, rounds):
    import torch
    n = 4096
    for scene in SCENES:
        arms = {'no sensor': _env(scene, n), '+ 32-ray sensor': _env(scene, n, dict(rays=_sensor(scene, 32)))}
        act = _actions(arms['no sensor'])
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
                    for k in range(len(eng.rays)):
                        eng.sense_rays(sensor=k)
                b.record()
                b.synchronize()
                if r:
                    res[label].append(a.elapsed_time(b) / steps)
        base = np.median(res['no sensor'])
        say('  {} x 4096 envs:'.format(scene))
        for label, v in res.items():
            say('    {:<16}: {:.3f} ms / step median of {} windows x {} steps (min {:.3f}, max {:.3f}); {:+.3f} ms '
                '= {:+.1f} % vs no sensor'.format(label, np.median(v), rounds, steps, min(v), max(v),
                                                  np.median(v) - base, 100 * (np.median(v) - base) / base))
        del arms
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
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r09_ray_sensor_cost.txt'))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('ray_sensor_cost.py needs a CUDA device')
    say('card: {}'.format(_card()))
    say('1. kernels alone, 4096 envs')
    kernels(args.launches)
    say('2. 4096 envs, device-resident: step + frames, the sensor cast behind the step')
    step_with_sensor(args.steps, args.rounds)
    if args.parent:
        say('3. bench.py (4096 falling_balls20 envs, no sensor): parent vs this tree, alternated in this run')
        bench_ab(os.path.abspath(args.parent), args.bench_rounds)
    say('card: {}'.format(_card()))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write('\n'.join(_LINES) + '\n')


if __name__ == '__main__':
    main()
