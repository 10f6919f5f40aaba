"""The RawState observer (moog/observers/raw_state.py:17-19): every sprite slot's state as float32
[N, S, 16], gathered from the state record by `moog_observe_sprites` (include/moog_b200.h).

The reference below (`project`) restates the layout of include/moog_b200_program.h (MOOG_OBS_*) in
numpy: the CUDA observation must equal it bit for bit (NaN as NaN) on the device record, and stay
within the parity bars of the step on the reference's recorded states.
"""
import ctypes
import os
import re

import numpy as np
import pytest

from tests import util

# (array, row) of the record behind columns 0-13 (include/moog_b200_program.h MOOG_OBS_*)
SOURCES = [('dyn', 0), ('dyn', 1), ('meta', 0), ('dyn', 4), ('stat', 1), ('stat', 2), ('stat', 6), ('stat', 7),
           ('stat', 8), ('stat', 9), ('dyn', 2), ('dyn', 3), ('dyn', 5), ('stat', 0)]
LAYER, ALIVE = 14, 15


def slot_layers(prog):
    """[S] layer index of every slot."""
    out = np.zeros(prog.n_slots, dtype=np.int64)
    for l in range(prog.n_layers):
        out[prog.layer_off[l]:prog.layer_off[l + 1]] = l
    return out


def project(prog, rec):
    """float32 [N, S, 16] of a state record (dict of numpy arrays with a leading env axis)."""
    N, S = rec['dyn'].shape[0], prog.n_slots
    layer = slot_layers(prog)
    first = np.asarray(prog.layer_off[:-1], dtype=np.int64)[layer]
    live = (np.arange(S) - first)[None, :] < rec['cnt'][:, layer]
    out = np.zeros((N, S, 16), dtype=np.float32)
    with np.errstate(over='ignore'):          # doubles beyond float32's range round to inf, as on the device
        for c, (k, row) in enumerate(SOURCES):
            out[:, :, c] = rec[k][:, row, :].astype(np.float32)
    out[~live] = 0.0
    out[:, :, LAYER] = layer
    out[:, :, ALIVE] = live
    return out


def bits_equal(a, b):
    """Equal bit for bit, except that any NaN equals any NaN."""
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    keep = ~np.isnan(a)
    return np.array_equal(a.view(np.uint32)[keep], b.view(np.uint32)[keep])


def within_parity(got, want64):
    """float32 observation vs the reference's float64 values: within util.RTOL (util.rel_err's floor)
    plus one float32 ulp; NaN and infinities identical."""
    got = np.asarray(got, dtype=np.float32)
    want32 = np.asarray(want64).astype(np.float32)
    fin = np.isfinite(want32)
    if not bits_equal(np.where(fin, 0, got), np.where(fin, 0, want32)):
        return False
    w = np.asarray(want64, dtype=np.float64)[fin]
    tol = util.RTOL * np.maximum(np.abs(w), util.ATOL_FLOOR / util.RTOL) + np.spacing(np.abs(want32[fin]))
    return bool((np.abs(got[fin].astype(np.float64) - w) <= tol).all())


def _config(name, raw_state=True, **level):
    import importlib
    import moog_b200  # noqa: F401
    from moog import observers
    mod = importlib.import_module('moog_b200.configs.' + name)
    cfg = mod.get_config(level or None)
    if raw_state:
        cfg['observers'] = dict(cfg['observers'], state=observers.RawState())
    return mod, cfg


# ---------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------

def test_compiler_records_the_raw_state_key():
    _, cfg = _config('falling_balls20', raw_state=False)
    from moog import observers
    from moog_b200 import compiler
    states = [cfg['state_initializer']()]
    assert compiler.compile_config(cfg, states).state_key is None
    cfg['observers'] = dict(cfg['observers'], sprites=observers.RawState())
    prog = compiler.compile_config(cfg, states)
    assert prog.state_key == 'sprites'
    cfg['observers']['more'] = observers.RawState()
    with pytest.raises(compiler.CompileError, match='only one RawState'):
        compiler.compile_config(cfg, states)


def test_observation_columns_match_the_header():
    from moog_b200 import compiler
    with open(os.path.join(util.ROOT, 'include', 'moog_b200_program.h')) as f:
        defs = dict(re.findall(r'#define MOOG_OBS_(\w+) (\d+)', f.read()))
    assert len(defs) == 17
    for name, value in defs.items():
        assert getattr(compiler, 'OBS_' + name) == int(value), name
    assert (compiler.OBS_LAYER, compiler.OBS_ALIVE) == (LAYER, ALIVE) and len(SOURCES) == compiler.OBS_MASS + 1


def test_observe_sprites_refuses_null_arguments_without_a_gpu():
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    L = capi.lib()
    st = capi.MoogState()
    buf = ctypes.c_void_p(16)
    assert L.moog_observe_sprites(None, ctypes.byref(st), 1, buf, None) == -1
    assert L.moog_observe_sprites(None, None, 0, None, None) == -1


# ---------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------

def _observe(eng):
    import torch
    out = torch.full((eng.n, eng.program.n_slots, 16), 7.0, dtype=torch.float32, device=eng.device)
    return eng.observe_sprites(out=out).cpu().numpy()


def _check_against_reference(prog, got, ref, exact, what):
    """got: [S, 16] observation of one env; ref: that env's recorded reference state (batch of 1)."""
    want = project(prog, ref)[0]
    if exact:
        assert bits_equal(got, want), what
        return
    live = want[:, ALIVE] == 1
    assert bits_equal(got[~live], want[~live]), what + ' empty slots'
    for c in (2, LAYER, ALIVE):
        assert bits_equal(got[:, c], want[:, c]), (what, c)
    for c, (k, row) in enumerate(SOURCES):
        if c != 2:
            assert within_parity(got[live, c], ref[k][0, row, live]), (what, c)


@pytest.mark.gpu
@pytest.mark.parametrize('scene', util.SCENES)
def test_observation_follows_reference_trajectory(scene):
    """Along the golden trajectory (as test_cuda_follows_reference_trajectory steps it): after the reset
    and after every step the observation is the projection of the device record, bit for bit, and of
    the reference's recorded state (bit for bit on the IEEE-exact scenes, else within the step's bars)."""
    from moog_b200.batched_env import Engine
    g = util.load_golden(scene)
    prog = g['program']
    eng = Engine(prog, 1, 'cuda:0')
    eng.state.upload(util.state_at(g, None, prefix='init'))
    eng.post_reset(rule_noise=util.reset_rule_noise(g))
    assert eng.sprites is None                  # the stored program has no RawState observer
    got = _observe(eng)
    assert bits_equal(got, project(prog, eng.state.download())), (scene, 'reset')
    _check_against_reference(prog, got[0], util.state_at(g, -1), True, '{} reset'.format(scene))
    exact = scene in util.EXACT_SCENES
    for t in range(len(g['reward'])):
        noise = g['noise'][t][None] if prog.noise_dim else None
        eng.env_step(g['actions'][t][None], noise=noise, rule_noise=util.rule_noise_at(g, t), auto_reset=False)
        got = _observe(eng)
        dev = eng.state.download()
        assert bits_equal(got, project(prog, dev)), (scene, t)
        _check_against_reference(prog, got[0], util.state_at(g, t), exact, '{} step {}'.format(scene, t))
        if not exact:                           # one step compared at a time, as the parity test does
            st = util.state_at(g, t)
            st['envi'], st['envf'] = dev['envi'], dev['envf']
            st['meta'][:, 1, :] |= dev['meta'][:, 1, :] & 64
            eng.state.upload(st)


@pytest.mark.gpu
def test_stale_slots_never_show():
    """NaN and garbage written into the record's empty slots after a step: those slots still read 0 in
    every column but the layer index."""
    import torch
    from moog_b200.batched_env import Engine
    g = util.load_golden('portal_zoo')
    prog = g['program']
    N = 97
    rng = np.random.RandomState(3)
    arrays = util.tile_state(util.state_at(g, -1), N)
    for l in range(prog.n_layers):
        arrays['cnt'][:, l] = rng.randint(0, arrays['cnt'][0, l] + 1, size=N)
    eng = Engine(prog, N, 'cuda:0')
    eng.state.upload(arrays)
    eng.env_step(None, auto_reset=False)
    dead = torch.from_numpy(~project(prog, eng.state.download())[:, :, ALIVE].astype(bool)).to('cuda:0')
    assert dead.any() and (~dead).any()
    st = eng.state
    for t, bad in ((st.dyn, float('nan')), (st.stat, -3.0e300), (st.meta, 0x7ffffff0)):
        t.copy_(torch.where(dead[:, None, :], torch.full_like(t, bad), t))
    got = _observe(eng)
    want = project(prog, st.download())
    assert bits_equal(got, want)
    d = dead.cpu().numpy()
    assert (got[d][:, :LAYER] == 0).all() and (got[d][:, ALIVE] == 0).all()
    assert not np.signbit(got[d][:, :LAYER]).any()


def _spawn_env(raw_state=True, seed=21, N=192):
    import torch
    from moog_b200.batched_env import BatchedEnvironment
    mod, cfg = _config('spawn_zoo', raw_state)
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(6)]
    env = BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=seed, initial_states=states,
                             layer_capacity=mod.LAYER_CAPACITY)
    ts = env.reset()
    env.engine.state.envi[:, 0] = torch.from_numpy(np.random.RandomState(4).randint(0, 40, size=N)).to(
        'cuda:0', dtype=torch.int32)       # staggered time-outs: auto-resets at many steps
    return env, ts


def _spawn_actions(T=140, N=192):
    rng = np.random.RandomState(5)
    return [rng.uniform(-1, 1, size=(N, 2)) for _ in range(T)]


@pytest.mark.gpu
def test_public_api_observation_with_auto_resets():
    """spawn_zoo (CreateSprites changes sprite counts mid-episode) with a RawState observer, 192 envs x
    140 steps through auto-resets: step() returns the projection of the record every step, FIRST steps
    included; twins with the same seed get byte-identical observations through step_to_host (every
    transport) and HostPipeline(depth=2) (both transports)."""
    import torch
    env, ts = _spawn_env()
    prog = env.program
    assert bits_equal(ts.observation['state'].cpu().numpy(), project(prog, env.engine.state.download()))
    acts = _spawn_actions()
    ref, firsts = [], 0
    for a in acts:
        ts = env.step(a)
        assert ts.observation['state'] is env.engine.sprites
        obs = ts.observation['state'].cpu().numpy()
        assert bits_equal(obs, project(prog, env.engine.state.download()))
        firsts += int((ts.step_type == 0).sum())
        ref.append(obs)
    assert firsts > 192, 'auto-resets happen during the run'
    assert max(int(o[:, :, ALIVE].sum()) for o in ref) > min(int(o[:, :, ALIVE].sum()) for o in ref)
    pin = lambda t: torch.empty(t.shape, dtype=t.dtype).pin_memory()
    for mode in ('mapped', 'device', 'chunked'):
        twin, _ = _spawn_env()
        e = twin.engine
        host = type(ts)(pin(e.step_type), pin(e.reward), pin(e.discount),
                        {'image': pin(e.frames), 'state': pin(e.sprites)})
        for k, a in enumerate(acts):
            out = twin.step_to_host(a, host, frames=mode)
            assert np.array_equal(out.observation['state'].numpy().view(np.uint32), ref[k].view(np.uint32)), (mode, k)
    for mode in ('mapped', 'device'):
        twin, _ = _spawn_env()
        pipe = twin.host_pipeline(depth=2, frames=mode)
        got = []
        for k, a in enumerate(acts):
            if k >= 2:
                got.append(pipe.collect().observation['state'].clone())
            pipe.submit(a)
        while len(got) < len(acts):
            got.append(pipe.collect().observation['state'].clone())
        for k, o in enumerate(got):
            assert np.array_equal(o.numpy().view(np.uint32), ref[k].view(np.uint32)), ('pipeline', mode, k)


@pytest.mark.gpu
@pytest.mark.parametrize('scene, n_envs', [('synthetic32', 131072), ('falling_balls20', 4097)])
def test_observation_at_size(scene, n_envs):
    """A full-size batch and one whose env count is not a multiple of the kernel's envs per CTA: the
    observation of a sample of envs (the last one included) is the projection of their records."""
    import torch
    from moog_b200.batched_env import BatchedEnvironment
    _, cfg = _config(scene)
    if scene == 'synthetic32':
        cfg['observers'] = {'state': cfg['observers']['state']}      # state only, as bench.py --state-only
    np.random.seed(9)
    states = [cfg['state_initializer']() for _ in range(64)]
    env = BatchedEnvironment(**cfg, num_envs=n_envs, device='cuda:0', seed=2, initial_states=states)
    env.reset()
    rng = np.random.RandomState(1)
    for _ in range(3):
        ts = env.step(torch.from_numpy(rng.randint(0, 5, size=(n_envs, 1)).astype(np.float64)))   # Grid
    idx = np.unique(np.concatenate([[0, 1, 2, 3, 4, n_envs - 2, n_envs - 1], rng.randint(0, n_envs, size=200)]))
    ti = torch.from_numpy(idx).to('cuda:0')
    st = env.engine.state
    rec = {k: getattr(st, k).index_select(0, ti).cpu().numpy() for k in ('dyn', 'stat', 'meta', 'cnt')}
    assert bits_equal(ts.observation['state'].index_select(0, ti).cpu().numpy(), project(env.program, rec))


@pytest.mark.gpu
def test_nothing_else_changes():
    """Frames are byte-identical with and without a RawState observer, the observer costs exactly one
    launch per step and a program without one allocates and launches nothing for it; VectorGymWrapper
    reports the space and returns the tensor."""
    import torch
    from moog_b200 import capi
    from moog_b200.env_wrappers import VectorGymWrapper
    plain, ts_p = _spawn_env(raw_state=False)
    raw, ts_r = _spawn_env(raw_state=True)
    assert plain.engine.sprites is None and set(ts_p.observation) == {'image'}
    assert set(ts_r.observation) == {'image', 'state'}
    for k, a in enumerate(_spawn_actions(T=60)):
        c0 = capi.launch_count()
        tp = plain.step(a)
        c1 = capi.launch_count()
        tr = raw.step(a)
        c2 = capi.launch_count()
        assert (c2 - c1) - (c1 - c0) == 1, k
        assert torch.equal(tp.observation['image'], tr.observation['image']), k
        assert torch.equal(tp.step_type, tr.step_type), k
    gym = VectorGymWrapper(raw)
    space = gym.observation_space['state']
    assert space == dict(low=-np.inf, high=np.inf, shape=(raw.program.n_slots, 16), dtype='float32')
    assert 'state' not in VectorGymWrapper(plain).observation_space
    obs, _, _, _ = gym.step(_spawn_actions(T=1)[0])
    assert obs['state'].shape == (192,) + space['shape'] and obs['state'].dtype == torch.float32
    assert bits_equal(obs['state'].cpu().numpy(), project(raw.program, raw.engine.state.download()))
    names = raw.shape_names()
    assert names and all(isinstance(n, str) for n in names)
