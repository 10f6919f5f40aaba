"""RaySensor: range-finder rays from an agent sprite to the first outline they cross.

The oracle is a plain numpy statement of the definition in moog/observers/pil_renderer.py RaySensor: slots
in ascending order, each slot's edges in outline order, every formula in float64 as written, a hit kept
when its t is <= the best so far (so the smallest t wins and a tie goes to the later slot), and a slot
that holds the origin by the even-odd rule reading t = 0 after its edges.

Without a GPU: the spec, the compiler, the gym space and the oracle against hand-worked cases.  On the
GPU: moog_ray_sensor and every BatchedEnvironment path against the oracle, float32 bit for bit.
"""
import ctypes
import importlib
import types

import numpy as np
import pytest

from tests import util

TWO_PI = 2 * np.pi


def _config(name, **observers):
    import moog_b200  # noqa: F401
    mod = importlib.import_module('moog_b200.configs.' + name)
    cfg = mod.get_config()
    if observers:
        cfg['observers'] = dict(cfg['observers'], **observers)
    return mod, cfg


def _sensor(*args, **kw):
    from moog import observers
    return observers.RaySensor(*args, **kw)


def _voff(prog):
    v = getattr(prog, 'voff', None)
    return np.asarray(v if v is not None and len(v) == prog.n_slots + 1 else util.prog_voff(prog))


def ray_oracle(prog, arrays, spec):
    """float32 [N, num_rays, 2]: the RaySensor readings of `spec` (a compiler ray dict) on `arrays`."""
    voff = _voff(prog)
    N, S = arrays['dyn'].shape[0], arrays['dyn'].shape[2]
    R, max_range = spec['num_rays'], spec['max_range']
    dx, dy = spec['dirs'][None, :, 0], spec['dirs'][None, :, 1]
    cnt, meta, vtx = arrays['cnt'], arrays['meta'], arrays['vtx']
    al, ai = spec['agent_layer'], spec['agent_index']
    agent = prog.layer_off[al] + ai
    has = cnt[:, al] > ai
    ox = np.where(has, arrays['dyn'][:, 0, min(agent, S - 1)], 0.0)[:, None]
    oy = np.where(has, arrays['dyn'][:, 1, min(agent, S - 1)], 0.0)[:, None]
    best = np.full((N, R), max_range)
    hit = np.full((N, R), -1)
    rows = np.arange(N)
    for l in range(prog.n_layers):
        for s in range(prog.layer_off[l], prog.layer_off[l + 1]):
            nv = meta[:, 2, s]
            target = has & (s - prog.layer_off[l] < cnt[:, l]) & bool((spec['layers'] >> l) & 1) & (s != agent)
            if not target.any():
                continue
            odd = np.zeros(N, dtype=bool)
            for j in range(int(nv[target].max(initial=0))):
                valid = (target & (j < nv))[:, None]
                a = vtx[rows, voff[s] + j]
                b = vtx[rows, voff[s] + np.where(j + 1 < nv, j + 1, 0)]
                ax, ay, bx, by = a[:, 0:1], a[:, 1:2], b[:, 0:1], b[:, 1:2]
                with np.errstate(all='ignore'):
                    ex, ey = bx - ax, by - ay
                    wx, wy = ax - ox, ay - oy
                    den = dx * ey - dy * ex
                    t = (wx * ey - wy * ex) / den
                    u = (wx * dy - wy * dx) / den
                    ok = valid & (den != 0) & (u >= 0) & (u <= 1) & (t >= 0) & (t <= best)
                    cross = ((ay > oy) != (by > oy)) & (ox < ax + (oy - ay) * (bx - ax) / (by - ay))
                best = np.where(ok, t, best)
                hit = np.where(ok, s, hit)
                odd ^= (valid & cross)[:, 0]
            best[odd] = 0.0
            hit[odd] = s
    out = np.empty((N, R, 2), dtype=np.float32)
    with np.errstate(all='ignore'):
        out[..., 0] = np.where(hit >= 0, (best / max_range).astype(np.float32), np.float32(1.0))
    out[..., 1] = hit.astype(np.float32)
    return out


# ---------------------------------------------------------------------------------------------
# hand-worked scenes: layer 0 holds the agent (slot 0, and a layer-mate in slot 1), layer 1 the targets
# ---------------------------------------------------------------------------------------------

def _square(cx, cy, h):
    return [(cx - h, cy - h), (cx + h, cy - h), (cx + h, cy + h), (cx - h, cy + h)]


def _scene(agent_xy, mates=(), targets=(), agent_outline=None):
    """(prog, arrays) of one env: slot 0 the agent at agent_xy, then its layer-mates, then the targets;
    every outline given as a list of vertices (the agent's defaults to a tiny square around it)."""
    outlines = [agent_outline or _square(agent_xy[0], agent_xy[1], 0.01)] + list(mates) + list(targets)
    S = len(outlines)
    voff = np.concatenate([[0], np.cumsum([len(o) for o in outlines])]).astype(int)
    names = ['agents', 'targets']
    prog = types.SimpleNamespace(n_layers=2, n_slots=S, layer_off=[0, 1 + len(mates), S], voff=list(voff),
                                 layer_names=names, layer_index=names.index)
    dyn = np.zeros((1, 6, S))
    meta = np.zeros((1, 3, S), dtype=np.int32)
    vtx = np.zeros((1, int(voff[-1]), 2))
    for s, o in enumerate(outlines):
        o = np.asarray(o, dtype=np.float64)
        vtx[0, voff[s]:voff[s + 1]] = o
        meta[0, 2, s] = len(o)
        dyn[0, :2, s] = o.mean(axis=0)
    dyn[0, :2, 0] = agent_xy
    cnt = np.zeros((1, 16), dtype=np.int32)
    cnt[0, 0], cnt[0, 1] = 1 + len(mates), len(targets)
    return prog, dict(dyn=dyn, meta=meta, vtx=vtx, cnt=cnt)


def _spec(prog, agent_layer='agents', **kw):
    from moog_b200 import compiler as C
    return C._lower_rays(prog, 'rays', _sensor(agent_layer, **kw))  # pylint: disable=protected-access


def _read(prog, arrays, **kw):
    return ray_oracle(prog, arrays, _spec(prog, **kw))[0]


def test_oracle_square_at_a_known_distance():
    prog, st = _scene((0.5, 0.5), targets=[_square(0.8, 0.5, 0.1)])
    # one ray with fov 2 pi points along `direction`: phi_0 = direction - pi + 2 pi * 0.5
    one = _read(prog, st, num_rays=1, direction=0.0, max_range=0.5)
    assert one[0, 1] == 1 and abs(one[0, 0] - 0.2 / 0.5) < 1e-6
    far = _read(prog, st, num_rays=1, direction=0.0, max_range=0.15)     # beyond max_range
    assert far.tolist() == [[1.0, -1.0]]
    back = _read(prog, st, num_rays=1, direction=np.pi, max_range=0.5)   # the square is behind
    assert back.tolist() == [[1.0, -1.0]]
    # four rays along -y, +x, +y and -x: only the second meets the square
    four = _read(prog, st, num_rays=4, direction=np.pi / 4, max_range=1.0)
    assert four[:, 1].tolist() == [-1.0, 1.0, -1.0, -1.0] and abs(four[1, 0] - 0.2) < 1e-6


def test_oracle_ray_through_a_vertex():
    diamond = [(0.7, 0.5), (0.8, 0.4), (0.9, 0.5), (0.8, 0.6)]
    prog, st = _scene((0.5, 0.5), targets=[diamond])
    got = _read(prog, st, num_rays=1, direction=0.0, max_range=1.0)
    assert got[0, 1] == 1 and abs(got[0, 0] - 0.2) < 1e-6


def test_oracle_edge_parallel_to_the_ray():
    # a flat outline lying on the ray: both its edges are parallel to the ray, den = 0, no hit
    flat = [(0.6, 0.5), (0.8, 0.5)]
    prog, st = _scene((0.5, 0.5), targets=[flat])
    assert _read(prog, st, num_rays=1, direction=0.0, max_range=1.0).tolist() == [[1.0, -1.0]]
    # a square whose bottom edge lies on the ray: that edge never hits, the left one does (u = 1)
    prog, st = _scene((0.5, 0.5), targets=[[(0.7, 0.5), (0.9, 0.5), (0.9, 0.7), (0.7, 0.7)]])
    got = _read(prog, st, num_rays=1, direction=0.0, max_range=1.0)
    assert got[0, 1] == 1 and abs(got[0, 0] - 0.2) < 1e-6


def test_oracle_origin_inside_reads_zero():
    prog, st = _scene((0.5, 0.5), targets=[_square(0.5, 0.5, 0.2), _square(0.55, 0.5, 0.01)])
    got = _read(prog, st, num_rays=8, max_range=0.5)
    # slot 1 holds the origin; slot 2 lies inside it, later in draw order, and is met at t > 0
    assert got[:, 0].tolist() == [0.0] * 8 and got[:, 1].tolist() == [1.0] * 8


def test_oracle_agent_excluded_and_layer_mates_hit():
    # the agent's own outline holds the origin; its layer-mate to the right is what +x meets
    prog, st = _scene((0.5, 0.5), mates=[_square(0.8, 0.5, 0.1)], agent_outline=_square(0.5, 0.5, 0.05))
    got = _read(prog, st, num_rays=1, direction=0.0, max_range=1.0, layers=['agents'])
    assert got[0, 1] == 1 and abs(got[0, 0] - 0.2) < 1e-6
    assert _read(prog, st, num_rays=1, direction=np.pi, max_range=1.0).tolist() == [[1.0, -1.0]]
    # the layer-mate as the agent: slot 0 is now a target, and the ray from (0.8, 0.5) along -x meets
    # its right edge at x = 0.55
    st2 = {k: v.copy() for k, v in st.items()}
    st2['dyn'][0, :2, 1] = (0.8, 0.5)
    got = _read(prog, st2, num_rays=1, direction=np.pi, max_range=1.0, agent_index=1)
    assert got[0, 1] == 0 and abs(got[0, 0] - 0.25) < 1e-6


def test_oracle_empty_agent_layer_reads_no_hit():
    prog, st = _scene((0.5, 0.5), targets=[_square(0.5, 0.5, 0.3)])
    st['cnt'][0, 0] = 0
    got = _read(prog, st, num_rays=5, max_range=1.0)
    assert got.tolist() == [[1.0, -1.0]] * 5
    st['cnt'][0, 0] = 1
    assert _read(prog, st, num_rays=5, max_range=1.0, agent_index=1).tolist() == [[1.0, -1.0]] * 5


def test_oracle_tie_goes_to_the_later_slot():
    prog, st = _scene((0.5, 0.5), targets=[_square(0.8, 0.5, 0.1), _square(0.8, 0.5, 0.1)])
    got = _read(prog, st, num_rays=1, direction=0.0, max_range=1.0)
    assert got[0, 1] == 2 and abs(got[0, 0] - 0.2) < 1e-6


# ---------------------------------------------------------------------------------------------
# the spec and the compiler, without a GPU
# ---------------------------------------------------------------------------------------------

def test_spec_defaults_and_direction_table():
    from moog_b200 import compiler as C
    s = _sensor('agent')
    assert (s._num_rays, s._max_range, s._fov, s._direction, s._layers, s._agent_index) == (
        32, 0.5, TWO_PI, np.pi / 2, None, 0)
    _, cfg = _config('colliding_predators84')
    np.random.seed(2)
    states = [cfg['state_initializer']()]
    prog = C.compile_config(dict(cfg, observers=dict(cfg['observers'], rays=s)), states)
    (key, r), = prog.rays
    assert key == 'rays' and r['agent_layer'] == prog.layer_index('agent') and r['agent_index'] == 0
    assert r['layers'] == (1 << prog.n_layers) - 1 and r['num_rays'] == 32 and r['max_range'] == 0.5
    k = np.arange(32)
    phi = np.pi / 2 - TWO_PI / 2 + TWO_PI * (k + 0.5) / 32
    assert r['dirs'].dtype == np.float64 and r['dirs'].shape == (32, 2) and r['dirs'].flags.c_contiguous
    assert np.array_equal(r['dirs'], np.stack([np.cos(phi), np.sin(phi)], axis=1))
    sub = C._lower_rays(prog, 'x', _sensor('predators', layers=['walls', 'agent'], agent_index=2,  # pylint: disable=protected-access
                                           num_rays=7, fov=np.pi / 3, direction=0.25, max_range=2))
    assert sub['layers'] == (1 << prog.layer_index('walls')) | (1 << prog.layer_index('agent'))
    assert sub['agent_index'] == 2 and sub['max_range'] == 2.0
    assert np.array_equal(sub['dirs'][:, 0], np.cos(0.25 - np.pi / 6 + np.pi / 3 * (np.arange(7) + 0.5) / 7))


@pytest.mark.parametrize('kw, what', [
    (dict(agent_layer='nobody'), "layer 'nobody'"),
    (dict(agent_layer='agent', layers=['walls', 'ghosts']), "layer 'ghosts'"),
    (dict(agent_layer='agent', num_rays=0), 'num_rays'),
    (dict(agent_layer='agent', num_rays=257), 'num_rays'),
    (dict(agent_layer='agent', num_rays=2.5), 'num_rays'),
    (dict(agent_layer='agent', max_range=0.0), 'max_range'),
    (dict(agent_layer='agent', max_range=-1.0), 'max_range'),
    (dict(agent_layer='agent', max_range=float('inf')), 'max_range'),
    (dict(agent_layer='agent', max_range=float('nan')), 'max_range'),
    (dict(agent_layer='agent', fov=0.0), 'fov'),
    (dict(agent_layer='agent', fov=TWO_PI + 1e-9), 'fov'),
    (dict(agent_layer='agent', fov=float('nan')), 'fov'),
    (dict(agent_layer='agent', agent_index=-1), 'agent_index'),
])
def test_compiler_refuses_bad_sensors(kw, what):
    from moog_b200 import compiler as C
    _, cfg = _config('colliding_predators84')
    np.random.seed(2)
    states = [cfg['state_initializer']()]
    with pytest.raises(C.CompileError, match=r"observer 'eyes': RaySensor .*" + what):
        C.compile_config(dict(cfg, observers=dict(cfg['observers'], eyes=_sensor(**kw))), states)


def test_ninth_sensor_is_refused():
    from moog_b200 import compiler as C
    _, cfg = _config('colliding_predators84')
    np.random.seed(2)
    states = [cfg['state_initializer']()]
    eight = {'r%d' % k: _sensor('agent', num_rays=k + 1) for k in range(8)}
    prog = C.compile_config(dict(cfg, observers=eight), states)
    assert [k for k, _ in prog.rays] == list(eight) and [r['num_rays'] for _, r in prog.rays] == list(range(1, 9))
    with pytest.raises(C.CompileError, match=r"observer 'r8': at most 8 RaySensor"):
        C.compile_config(dict(cfg, observers=dict(eight, r8=_sensor('agent'))), states)


def test_key_order_without_renderer_and_blob_identity():
    from moog import observers
    from moog_b200 import compiler as C
    from moog.observers import polygon_modifiers
    _, cfg = _config('timed_center')
    np.random.seed(2)
    states = [cfg['state_initializer']()]
    layer = list(states[0].keys())[-1]
    obs = dict(r1=_sensor(layer, num_rays=3), image=cfg['observers']['image'], state=observers.RawState(),
               mask=observers.SpriteMask(image_size=(32, 32)), r0=_sensor(layer, num_rays=5),
               side=observers.PILRenderer(image_size=(48, 48), polygon_modifier=polygon_modifiers.DoNothing()))
    prog = C.compile_config(dict(cfg, observers=obs), states)
    assert [k for k, _ in prog.rays] == ['r1', 'r0'] and [r['num_rays'] for _, r in prog.rays] == [3, 5]
    assert [k for k, _ in prog.views] == ['image', 'side'] and [k for k, _ in prog.masks] == ['mask']
    assert prog.state_key == 'state'
    plain = C.compile_config(dict(cfg, observers={k: v for k, v in obs.items() if k[0] != 'r'}), states)
    assert prog.blob == plain.blob
    # a sensor alone: no renderer, and the blob of a config without observers
    _, cfg = _config('falling_balls20')
    np.random.seed(2)
    states = [cfg['state_initializer']()]
    only = C.compile_config(dict(cfg, observers={'rays': _sensor('balls', agent_index=3)}), states)
    assert only.render is None and only.views == [] and only.masks == [] and [k for k, _ in only.rays] == ['rays']
    assert only.blob == C.compile_config(dict(cfg, observers={}), states).blob
    # every config under configs/ with a sensor on its last layer compiles to its own bytes (those whose
    # state initializer needs no device here)
    import pkgutil
    import moog_b200.configs as configs
    from moog_b200 import capi
    checked = []
    for info in pkgutil.iter_modules(configs.__path__):
        mod, cfg = _config(info.name)
        np.random.seed(5)
        try:
            states = [cfg['state_initializer']() for _ in range(2)]
        except capi.MoogError:
            continue
        cap = getattr(mod, 'LAYER_CAPACITY', None)
        last = list(states[0].keys())[-1]
        with_rays = C.compile_config(dict(cfg, observers=dict(cfg['observers'], eyes=_sensor(last))), states, cap)
        assert with_rays.blob == C.compile_config(cfg, states, cap).blob, info.name
        checked.append(info.name)
    assert len(checked) >= 6, checked


def test_gym_observation_space():
    from moog_b200 import compiler as C
    from moog_b200.env_wrappers import VectorGymWrapper
    _, cfg = _config('colliding_predators84')
    np.random.seed(2)
    states = [cfg['state_initializer']()]
    prog = C.compile_config(dict(cfg, observers=dict(cfg['observers'], rays=_sensor('agent', num_rays=33))),
                            states)
    wrapper = object.__new__(VectorGymWrapper)
    wrapper._env = types.SimpleNamespace(program=prog)   # pylint: disable=protected-access
    spaces = wrapper.observation_space
    assert spaces['rays'] == dict(low=-1, high=max(1, prog.n_slots - 1), shape=(33, 2), dtype='float32')
    tiny = types.SimpleNamespace(views=[], masks=[], state_key=None, n_slots=1, rays=prog.rays)
    wrapper._env = types.SimpleNamespace(program=tiny)   # pylint: disable=protected-access
    assert wrapper.observation_space['rays']['high'] == 1


# ---------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------

def _states(g, steps):
    parts = [util.state_at(g, int(t)) for t in steps]
    return {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}


def _steps(g, k=4):
    T = len(g['reward'])
    return [-1] + [int(t) for t in np.linspace(0, T - 1, k - 1).round()]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def _scene_specs(prog):
    """Sensors over every combination the kernel distinguishes: ray counts around a warp, both fovs, a short and
    a long range, every agent layer, a layer subset and an agent index beyond the first."""
    from moog_b200 import compiler as C
    names = prog.layer_names
    specs = []
    for i, (R, fov, rng) in enumerate([(1, TWO_PI, 0.1), (7, np.pi / 3, 2.0), (32, TWO_PI, 2.0),
                                       (33, np.pi / 3, 0.1), (256, TWO_PI, 2.0)]):
        for l, name in enumerate(names):
            sub = [n for k, n in enumerate(names) if (k + i) % 2 == 0] or None
            for kw in (dict(), dict(layers=sub, agent_index=1 + (i % 2))):
                specs.append(C._lower_rays(prog, 's', _sensor(  # pylint: disable=protected-access
                    name, num_rays=R, fov=fov, max_range=rng, direction=0.3 * i + 0.1 * l, **kw)))
    return specs


@pytest.mark.gpu
@pytest.mark.parametrize('scene', util.SCENES)
def test_ray_kernel_matches_oracle(scene):
    """moog_ray_sensor on states across the golden trajectory, for every sensor of _scene_specs: float32 bits
    equal to the oracle's; and a range into pinned host memory."""
    import torch
    from moog_b200.batched_env import Engine
    g = util.load_golden(scene)
    prog = g['program']
    arrays = _states(g, _steps(g))
    specs = _scene_specs(prog)
    checked = 0
    for base in range(0, len(specs), 8):
        prog.rays = [('s%d' % k, r) for k, r in enumerate(specs[base:base + 8])]
        eng = Engine(prog, arrays['dyn'].shape[0], 'cuda:0')
        eng.state.upload(arrays)
        for k, (_, r) in enumerate(prog.rays):
            got = eng.sense_rays(sensor=k).cpu().numpy()
            want = ray_oracle(prog, arrays, r)
            assert got.shape == want.shape == (arrays['dyn'].shape[0], r['num_rays'], 2)
            assert np.array_equal(_bits(got), _bits(want)), (scene, base + k, r['num_rays'], r['agent_layer'])
            checked += 1
    assert checked == len(specs)
    host = torch.full(eng.rays[0].shape, 7.0, dtype=torch.float32).pin_memory()
    eng.sense_rays(out=host, first=2, count=eng.n - 2, sensor=0)
    torch.cuda.synchronize()
    assert torch.equal(host[2:], eng.rays[0][2:].cpu()) and bool((host[:2] == 7).all())


def _env(cfg, mod, N, seed, states, observers, reset_mode='pool', age=0, start=True):
    import torch
    from moog_b200.batched_env import BatchedEnvironment
    np.random.seed(11)
    env = BatchedEnvironment(**dict(cfg, observers=observers), num_envs=N, device='cuda:0', seed=seed,
                             initial_states=states, layer_capacity=getattr(mod, 'LAYER_CAPACITY', None),
                             reset_mode=reset_mode)
    if not start:
        return env, None
    ts = env.reset()
    env.engine.state.envi[:, 0] = torch.from_numpy(np.random.RandomState(4).randint(age, age + 30, size=N)).to(
        'cuda:0', dtype=torch.int32)       # staggered time-outs: auto-resets at many steps
    return env, ts


def _actions(env, T, seed=5):
    rng = np.random.RandomState(seed)
    width = env.action_dim
    if width == 1:   # Grid
        return [rng.randint(0, 5, size=(env.num_envs, 1)).astype(np.float64) for _ in range(T)]
    return [rng.uniform(-1, 1, size=(env.num_envs, width)) for _ in range(T)]


ENV_CASES = [('colliding_predators84', 'device', 150, dict(agent_layer='agent')),
             ('spawn_zoo', 'pool', 0, dict(agent_layer='agent', layers=['drops', 'sparks', 'walls'])),
             ('falling_balls20', 'pool', 0, dict(agent_layer='balls', agent_index=3))]


@pytest.mark.gpu
@pytest.mark.parametrize('name, reset_mode, age, origin', ENV_CASES)
def test_environment_rays_match_oracle(name, reset_mode, age, origin):
    """A BatchedEnvironment with two RaySensors stepped 100 times through auto-resets: every step's readings
    equal the oracle's on the downloaded state, and the frames, a mask and the RawState equal those of a twin
    without sensors."""
    import torch
    from moog import observers
    mod, cfg = _config(name)
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(6)]
    N, T = 12, 100
    base = dict(cfg['observers'], state=observers.RawState(), mask=observers.SpriteMask(image_size=(48, 48)))
    obs = dict(base, near=_sensor(num_rays=32, max_range=0.3, **origin),
               wide=_sensor(num_rays=33, max_range=1.5, fov=np.pi / 3, direction=1.0, **origin))
    env, ts = _env(cfg, mod, N, 7, states, obs, reset_mode, age)
    twin, ts_t = _env(cfg, mod, N, 7, states, base, reset_mode, age)
    prog = env.program
    acts = _actions(env, T)
    firsts = hits = 0
    for t in range(T + 1):
        if t > 0:
            ts, ts_t = env.step(acts[t - 1]), twin.step(acts[t - 1])
        for key in ('image', 'state', 'mask'):
            assert torch.equal(ts.observation[key], ts_t.observation[key]), (name, key, t)
        arrays = env.engine.state.download()
        for k, key in enumerate(('near', 'wide')):
            got = ts.observation[key].cpu().numpy()
            want = ray_oracle(prog, arrays, prog.rays[k][1])
            assert np.array_equal(_bits(got), _bits(want)), (name, key, t)
            hits += int((got[..., 1] >= 0).sum())
        firsts += int((ts.step_type == 0).sum())
    assert firsts > N, 'auto-resets happen during the run'
    assert hits > 0, 'the rays meet sprites'
    assert torch.equal(env.observation()['wide'], ts.observation['wide'])


def _clone(ts):
    return type(ts)(ts.step_type.clone(), ts.reward.clone(), ts.discount.clone(),
                    {k: v.clone() for k, v in ts.observation.items()})


@pytest.mark.gpu
@pytest.mark.parametrize('n_envs', [4096, 1001])
def test_rays_through_every_transport(n_envs):
    """falling_balls20 with a 32-ray and a 7-ray sensor (56 bytes per env: cast whole under 'chunked') and a
    RawState: step_to_host ('mapped', 'device', 'chunked') and HostPipeline(depth=2) ('mapped', 'device')
    deliver what step() returns."""
    import torch
    from moog import observers
    mod, cfg = _config('falling_balls20')
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(16)]
    obs = dict(cfg['observers'], state=observers.RawState(), rays=_sensor('balls', num_rays=32),
               odd=_sensor('balls', num_rays=7, agent_index=5, max_range=1.0))
    keys = ('image', 'state', 'rays', 'odd')
    T = 12
    env, _ = _env(cfg, mod, n_envs, 21, states, obs, start=False)
    ts = env.reset()
    acts = _actions(env, T)
    ref = [{k: v.cpu().clone() for k, v in ts.observation.items()}]
    meta = [(ts.step_type.cpu().clone(), ts.reward.cpu().clone())]
    for a in acts:
        ts = env.step(a)
        assert set(ts.observation) == set(keys)
        assert ts.observation['rays'] is env.engine.rays[0]
        ref.append({k: v.cpu().clone() for k, v in ts.observation.items()})
        meta.append((ts.step_type.cpu().clone(), ts.reward.cpu().clone()))

    def same(got, k, what):
        for key in keys:
            assert torch.equal(got.observation[key].cpu(), ref[k][key]), (what, key, k)
        assert torch.equal(got.step_type.cpu(), meta[k][0]), (what, k)
        assert torch.equal(got.reward.cpu().nan_to_num(-7.0), meta[k][1].nan_to_num(-7.0)), (what, k)

    pin = lambda t: torch.empty(t.shape, dtype=t.dtype).pin_memory()
    for mode in ('mapped', 'device', 'chunked'):
        twin, _ = _env(cfg, mod, n_envs, 21, states, obs, start=False)   # the first call is the reset
        e = twin.engine
        host = type(ts)(pin(e.step_type), pin(e.reward), pin(e.discount),
                        {'image': pin(e.frames), 'state': pin(e.sprites), 'rays': pin(e.rays[0]),
                         'odd': pin(e.rays[1])})
        same(twin.step_to_host(None, host, frames=mode), 0, mode)
        for k, a in enumerate(acts, 1):
            same(twin.step_to_host(a, host, frames=mode), k, mode)
    for mode in ('mapped', 'device'):
        twin, _ = _env(cfg, mod, n_envs, 21, states, obs, start=False)
        pipe = twin.host_pipeline(depth=2, frames=mode)
        seq = [None] + acts
        got = []
        for k, a in enumerate(seq):
            if k >= 2:
                got.append(_clone(pipe.collect()))
            pipe.submit(a)
        while len(got) < len(seq):
            got.append(_clone(pipe.collect()))
        for k, g in enumerate(got):
            same(g, k, 'pipeline ' + mode)


@pytest.mark.gpu
def test_launches_with_sensors():
    """M sensors launch exactly M more kernels per step; frames, state and rewards are those of the program
    without sensors."""
    import torch
    from moog_b200 import capi
    mod, cfg = _config('spawn_zoo')
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(6)]
    N = 256
    extra = dict(a=_sensor('agent', num_rays=1), b=_sensor('agent', num_rays=256), c=_sensor('walls', num_rays=40))
    one, _ = _env(cfg, mod, N, 3, states, cfg['observers'])
    many, _ = _env(cfg, mod, N, 3, states, dict(cfg['observers'], **extra))
    assert one.engine.rays == [] and len(many.engine.rays) == 3
    for k, a in enumerate(_actions(one, 40)):
        c0 = capi.launch_count()
        t1 = one.step(a)
        c1 = capi.launch_count()
        tm = many.step(a)
        c2 = capi.launch_count()
        assert (c2 - c1) - (c1 - c0) == len(extra), k
        assert torch.equal(t1.observation['image'], tm.observation['image']), k
        assert torch.equal(t1.step_type, tm.step_type), k
        assert torch.equal(t1.reward.nan_to_num(-7.0), tm.reward.nan_to_num(-7.0)), k


@pytest.mark.gpu
def test_bad_arguments_are_refused_and_launch_nothing():
    import torch
    from moog_b200 import capi
    from moog_b200.batched_env import Engine
    g = util.load_golden('colliding_predators')
    prog = g['program']
    prog.rays = [('s', _scene_specs(prog)[2])]
    arrays = _states(g, _steps(g))
    eng = Engine(prog, arrays['dyn'].shape[0], 'cuda:0')
    eng.state.upload(arrays)
    L = capi.lib()
    spec0, dirs = eng._ray_specs[0]   # pylint: disable=protected-access
    out = eng.rays[0]
    st = eng.state.struct()
    stream = eng._stream()   # pylint: disable=protected-access

    def call(spec=None, n=eng.n, dst=None, p=eng.dev_program.handle, state=ctypes.byref(st)):
        spec = spec0 if spec is None else spec
        return L.moog_ray_sensor(p, state, n, None if spec == 'null' else ctypes.byref(spec),
                                 ctypes.c_void_p(out.data_ptr()) if dst is None else dst, stream)

    def changed(**fields):
        s = capi.MoogRaySpec.from_buffer_copy(spec0)
        for k, v in fields.items():
            setattr(s, k, v)
        return s
    c0 = capi.launch_count()
    cases = [dict(p=None), dict(state=None), dict(spec='null'), dict(dst=ctypes.c_void_p(0)), dict(n=-1),
             dict(dst=ctypes.c_void_p(out.data_ptr() + 8)),
             dict(spec=changed(dirs=None)), dict(spec=changed(dirs=dirs.data_ptr() + 4)),
             dict(spec=changed(n_rays=0)), dict(spec=changed(n_rays=257)),
             dict(spec=changed(max_range=0.0)), dict(spec=changed(max_range=-1.0)),
             dict(spec=changed(max_range=float('inf'))), dict(spec=changed(max_range=float('nan'))),
             dict(spec=changed(agent_layer=-1)), dict(spec=changed(agent_layer=prog.n_layers)),
             dict(spec=changed(agent_index=-1)), dict(spec=changed(layers=1 << prog.n_layers)),
             dict(spec=changed(layers=0x80000000))]
    for kw in cases:
        assert call(**kw) == capi.E_INVAL, kw
    assert call(n=0) == 0
    assert capi.launch_count() == c0
    assert call() == 0 and capi.launch_count() == c0 + 1
    torch.cuda.synchronize()
    assert np.array_equal(_bits(out.cpu().numpy()), _bits(ray_oracle(prog, arrays, prog.rays[0][1])))
