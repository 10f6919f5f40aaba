"""Several PILRenderer observers per config (environment.py:118-126 fills every entry of `observers`):
view 0 is the first renderer and lives in the header words MOOG_H_R_*, every further renderer is a row
of the program's view table (include/moog_b200_program.h MOOG_H_VIEWS), drawn by `moog_render_view`.

Every view must be what the reference draws with that renderer's settings (the recorded anti-aliased
and large frames of tests/golden), and what a program with that renderer alone draws, through every
public path.
"""
import ctypes
import importlib
import os
import re

import numpy as np
import pytest

from tests import util


def _config(name, **observers):
    import moog_b200  # noqa: F401
    mod = importlib.import_module('moog_b200.configs.' + name)
    cfg = mod.get_config()
    if observers:
        cfg['observers'] = dict(cfg['observers'], **observers)
    return mod, cfg


def _renderer(**kw):
    from moog import observers
    return observers.PILRenderer(**kw)


def _torus(layers):
    from moog.observers import polygon_modifiers
    return polygon_modifiers.TorusGeometry(layers)


def with_views(blob, rows):
    """`blob` with a view table of `rows` (lists of MOOG_VIEW_WORDS ints) appended to its ipool -- the
    layout compiler.Program.finalize writes for a config with 1 + len(rows) renderers."""
    from moog_b200 import compiler as C
    b = bytes(bytearray(blob))
    hdr = np.frombuffer(b[:C.HDR_WORDS * 4], dtype='<i4').copy()
    n_ops, n_ipool = int(hdr[C.H_N_OPS]), int(hdr[C.H_N_IPOOL])
    start = C.HDR_WORDS * 4 + 80 * n_ops
    padded = (n_ipool + 1) & ~1
    ipool = list(np.frombuffer(b[start:start + 4 * n_ipool], dtype='<i4'))
    rest = b[start + 4 * padded:]
    hdr[C.H_VIEWS] = len(ipool)
    hdr[C.H_N_VIEWS] = len(rows)
    ipool += [int(w) for r in rows for w in r]
    hdr[C.H_N_IPOOL] = len(ipool)
    if len(ipool) % 2:
        ipool.append(0)
    out = b[C.HDR_WORDS * 4:start] + np.asarray(ipool, dtype='<i4').tobytes() + rest
    hdr[C.H_BYTES] = C.HDR_WORDS * 4 + len(out)
    return hdr.tobytes() + out


def _validate(blob):
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    buf = (ctypes.c_uint8 * len(blob)).from_buffer_copy(bytes(blob))
    return capi.lib().moog_program_validate(ctypes.cast(buf, ctypes.c_void_p), len(blob))


# ---------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------

def test_view_words_match_the_header():
    from moog_b200 import compiler as C
    with open(os.path.join(util.ROOT, 'include', 'moog_b200_program.h')) as f:
        text = f.read()
    defs = dict(re.findall(r'#define MOOG_(VIEW_WORDS|MAX_VIEWS) (\d+)', text))
    assert (C.VIEW_WORDS, C.MAX_VIEWS) == (int(defs['VIEW_WORDS']), int(defs['MAX_VIEWS'])) == (8, 8)
    assert (C.H_VIEWS, C.H_N_VIEWS) == tuple(int(v) for v in re.search(
        r'MOOG_H_VIEWS = (\d+),.*?MOOG_H_N_VIEWS = (\d+),', text, re.S).groups())
    assert C.H_R_ENABLED - C.H_R_HEIGHT + 1 == C.VIEW_WORDS
    # the words were free before: no stored program uses them
    for name in util.SCENES:
        hdr = np.frombuffer(bytes(bytearray(util.load_golden(name)['blob']))[:C.HDR_WORDS * 4], dtype='<i4')
        assert hdr[C.H_VIEWS] == 0 and hdr[C.H_N_VIEWS] == 0, name


def test_compiler_keeps_observer_order():
    from moog import observers
    from moog_b200 import compiler as C
    _, cfg = _config('timed_center')
    states = [cfg['state_initializer']()]
    one = C.compile_config(cfg, states)
    assert [k for k, _ in one.views] == ['image'] and one.render == one.views[0][1]
    assert one.header[C.H_VIEWS] == 0 and one.header[C.H_N_VIEWS] == 0
    cfg['observers'] = {'state': observers.RawState(),
                        'big': _renderer(image_size=(128, 96), bg_color=(10, 20, 30)),
                        'image': cfg['observers']['image'],
                        'torus': _renderer(anti_aliasing=2, color_to_rgb='hsv_to_rgb',
                                           polygon_modifier=_torus(['agent']))}
    prog = C.compile_config(cfg, states)
    assert prog.state_key == 'state'
    assert [k for k, _ in prog.views] == ['big', 'image', 'torus']
    assert prog.render is prog.views[0][1]
    assert (prog.render['width'], prog.render['height']) == (128, 96)
    hdr = prog.header
    assert hdr[C.H_N_VIEWS] == 2
    assert list(hdr[C.H_R_HEIGHT:C.H_R_ENABLED + 1]) == [96, 128, 1, 10 | 20 << 8 | 30 << 16, C.CMAP_NONE,
                                                         C.PMOD_NONE, 0, 1]
    n_ops = int(hdr[C.H_N_OPS])
    ipool = np.frombuffer(prog.blob[C.HDR_WORDS * 4 + 80 * n_ops:], dtype='<i4')
    table = ipool[hdr[C.H_VIEWS]:hdr[C.H_VIEWS] + 2 * C.VIEW_WORDS].reshape(2, C.VIEW_WORDS)
    agent = prog.layer_index('agent')
    assert list(table[0]) == [64, 64, 1, 0, C.CMAP_HSV, C.PMOD_FIRST_PERSON, agent, 1]
    assert list(table[1]) == [64, 64, 2, 0, C.CMAP_HSV, C.PMOD_TORUS, 0, 1]
    # view 0's words and everything before the table are those of the program with view 0 alone
    cfg['observers'] = {'state': observers.RawState(), 'big': cfg['observers']['big']}
    alone = C.compile_config(cfg, states)
    assert prog.blob[C.HDR_WORDS * 4:C.HDR_WORDS * 4 + 80 * n_ops] == alone.blob[C.HDR_WORDS * 4:C.HDR_WORDS * 4 + 80 * n_ops]
    assert _validate(prog.blob) == 0 and _validate(alone.blob) == 0
    cfg['observers'] = {'v%d' % k: _renderer() for k in range(C.MAX_VIEWS)}
    assert len(C.compile_config(cfg, states).views) == C.MAX_VIEWS
    cfg['observers']['one_more'] = _renderer()
    with pytest.raises(C.CompileError, match='at most 8 PILRenderer'):
        C.compile_config(cfg, states)


def test_view_table_is_validated():
    """moog_program_validate checks every row of the view table with the bounds of the header's
    renderer words, and the table itself."""
    from moog_b200 import compiler as C
    g = util.load_golden('timed_center')
    base = bytes(bytearray(g['blob']))
    hdr0 = np.frombuffer(base[:C.HDR_WORDS * 4], dtype='<i4')
    n_layers = int(hdr0[C.H_N_LAYERS])
    good_row = [64, 64, 1, 0, C.CMAP_HSV, C.PMOD_FIRST_PERSON, n_layers - 1, 1]
    rows = [good_row, [128, 128, 2, 0x102030, C.CMAP_NONE, C.PMOD_TORUS, 0, 1]]
    assert _validate(base) == 0
    assert _validate(with_views(base, rows)) == 0
    assert _validate(with_views(base, [good_row] * (C.MAX_VIEWS - 1))) == 0

    def bad_row(k, value):
        r = [list(x) for x in rows]
        r[1][k] = value
        return _validate(with_views(base, r))

    for k, v in ((0, 0), (0, 8193), (1, 0), (1, 8193), (2, 0), (2, 17), (4, 2), (4, -1), (5, 3), (5, -1), (7, 0)):
        assert bad_row(k, v) != 0, (k, v)
    r = [list(good_row)]
    r[0][6] = n_layers
    assert _validate(with_views(base, r)) != 0                          # FirstPersonAgent layer
    r[0][6] = -1
    assert _validate(with_views(base, r)) != 0
    assert _validate(with_views(base, [good_row] * C.MAX_VIEWS)) != 0   # 9 renderers

    def edit(blob, word, value):
        b = np.frombuffer(blob, dtype=np.uint8).copy()
        b[:C.HDR_WORDS * 4].view('<i4')[word] = value
        return b.tobytes()

    two = with_views(base, rows)
    n_ipool = int(np.frombuffer(two[:C.HDR_WORDS * 4], dtype='<i4')[C.H_N_IPOOL])
    assert _validate(edit(two, C.H_VIEWS, -1)) != 0                     # table outside ipool
    assert _validate(edit(two, C.H_VIEWS, n_ipool - C.VIEW_WORDS)) != 0
    assert _validate(edit(two, C.H_N_VIEWS, -1)) != 0
    assert _validate(edit(two, C.H_N_VIEWS, 3)) != 0                    # rows beyond ipool
    assert _validate(edit(two, C.H_R_ENABLED, 0)) != 0                  # further views need a view 0


def test_render_view_refuses_null_arguments_without_a_gpu():
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    L = capi.lib()
    st = capi.MoogState()
    buf = ctypes.c_void_p(16)
    for view in (0, 1, -1, 8):
        assert L.moog_render_view(None, ctypes.byref(st), 1, view, buf, None) == -1
    assert L.moog_render_view(None, None, 0, 0, None, None) == -1


# ---------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------

def _row(hdr, height=None, width=None, aa=None):
    from moog_b200 import compiler as C
    r = [int(w) for w in hdr[C.H_R_HEIGHT:C.H_R_ENABLED + 1]]
    for k, v in ((0, height), (1, width), (2, aa)):
        if v is not None:
            r[k] = v
    return r


def _stub(blob, layer_names, rows):
    prog = util.ProgramStub(with_views(blob, rows), layer_names)
    prog.views = [('image', prog.render)] + [('v%d' % k, dict(height=r[0], width=r[1], aa=r[2]))
                                             for k, r in enumerate(rows, 1)]
    return prog


@pytest.mark.gpu
@pytest.mark.parametrize('scene', sorted(set(util.AA_SCENES) | set(util.BIG_SCENES)))
def test_views_match_reference_frames(scene):
    """One program per scene whose views are the primary 64 x 64 renderer and the anti-aliased / large
    settings recorded from the reference (tests/golden/*_aa.npz, *_big.npz): every view drawn by
    moog_render_view from the recorded states, 0 differing bytes."""
    import torch
    from moog_b200 import compiler as C
    from moog_b200.batched_env import Engine
    g = util.load_golden(scene)
    hdr = np.frombuffer(bytes(bytearray(g['blob']))[:C.HDR_WORDS * 4], dtype='<i4')
    sets = []   # (golden of recorded frames, {view: key of its frames})
    rows = []
    if scene in util.AA_SCENES:
        sets.append((util.load_golden_aa(scene), {}))
        for aa in (2, 3):
            rows.append(_row(hdr, aa=aa))
            sets[-1][1][len(rows)] = 'frames_aa%d' % aa
    if scene in util.BIG_SCENES:
        sets.append((util.load_golden_big(scene), {}))
        for w, h in util.BIG_SIZES:
            rows.append(_row(hdr, height=h, width=w))
            sets[-1][1][len(rows)] = 'frames_%dx%d' % (w, h)
    prog = _stub(g['blob'], g['layer_names'], rows)
    for ref, views in sets:
        parts = [util.state_at(g, int(t)) for t in ref['frame_steps']]
        arrays = {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}
        eng = Engine(prog, arrays['dyn'].shape[0], 'cuda:0')
        eng.state.upload(arrays)
        assert eng.n_views == 1 + len(rows)
        for v, key in views.items():
            out = eng.render(view=v, out=torch.full_like(eng.view_buffer(v), 7)).cpu().numpy()
            assert out.shape == ref[key].shape, (scene, key)
            assert int((out != ref[key]).sum()) == 0, (scene, key)
        # view 0 through moog_render_view == moog_render
        a = eng.render(out=torch.zeros_like(eng.frames))
        b = eng.render(out=torch.full_like(eng.frames, 9))
        from moog_b200 import capi
        st = eng.state.struct()
        capi.check(capi.lib().moog_render_view(eng.dev_program.handle, ctypes.byref(st), eng.n, 0,
                                               ctypes.c_void_p(b.data_ptr()), eng._stream()))
        assert torch.equal(a, b), scene
        # bad view indices and a misaligned destination
        for bad in (-1, 1 + len(rows)):
            assert capi.lib().moog_render_view(eng.dev_program.handle, ctypes.byref(st), eng.n, bad,
                                               ctypes.c_void_p(b.data_ptr()), eng._stream()) == -1
        assert capi.lib().moog_render_view(eng.dev_program.handle, ctypes.byref(st), eng.n, 1,
                                           ctypes.c_void_p(b.data_ptr() + 4), eng._stream()) == -1
        torch.cuda.synchronize()


def _env(cfg, mod, N, seed, states, observers, reset_mode='pool', start=True, age=0):
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


# step_count the twins start from: every env reaches its config's time-out within the run
TWIN_AGE = {'timed_center': 0, 'colliding_predators84': 150, 'spawn_zoo': 0}
TWIN_CASES = {
    # FirstPersonAgent primary (the config's own) + an allocentric 128 x 128 view
    'timed_center': lambda: dict(alloc=_renderer(image_size=(128, 128), color_to_rgb='hsv_to_rgb')),
    # a TorusGeometry view, raw colours next to hsv, a non-default background
    'colliding_predators84': lambda: dict(
        torus=_renderer(image_size=(64, 64), color_to_rgb='hsv_to_rgb', polygon_modifier=_torus(['predators'])),
        raw=_renderer(image_size=(48, 40), bg_color=(40, 90, 200))),
    'spawn_zoo': lambda: dict(bg=_renderer(image_size=(96, 96), bg_color=(255, 255, 255), color_to_rgb='hsv_to_rgb')),
}


@pytest.mark.gpu
@pytest.mark.parametrize('name, reset_mode', [('timed_center', 'pool'), ('colliding_predators84', 'pool'),
                                              ('colliding_predators84', 'device'), ('spawn_zoo', 'pool')])
def test_every_view_equals_its_single_renderer_twin(name, reset_mode):
    """A multi-view BatchedEnvironment stepped ~100 times through auto-resets against one environment
    per renderer that has only that renderer (same seed, same actions): every view's frames, the
    state, reward and step_type bit-identical, FIRST steps included."""
    import torch
    mod, cfg = _config(name)
    extra = TWIN_CASES[name]()
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(6)]
    N, T = 160, 100
    multi, ts_m = _env(cfg, mod, N, 7, states, dict(cfg['observers'], **extra), reset_mode, age=TWIN_AGE[name])
    keys = ['image'] + list(extra)
    assert multi._image_keys == keys and multi.engine.n_views == len(keys)
    twins = {}
    for k in keys:
        twin, ts_t = _env(cfg, mod, N, 7, states, {k: dict(cfg['observers'], **extra)[k]}, reset_mode,
                          age=TWIN_AGE[name])
        twins[k] = (twin, ts_t)
    acts = _actions(multi, T)
    firsts = 0
    for t in range(T + 1):
        if t > 0:
            ts_m = multi.step(acts[t - 1])
        assert set(ts_m.observation) == set(keys)
        st_m = multi.engine.state
        for k in keys:
            twin, ts_t = twins[k]
            if t > 0:
                ts_t = twin.step(acts[t - 1])
            assert torch.equal(ts_m.observation[k], ts_t.observation[k]), (name, k, t)
            assert torch.equal(ts_m.step_type, ts_t.step_type), (name, k, t)
            assert torch.equal(ts_m.reward.nan_to_num(-7.0), ts_t.reward.nan_to_num(-7.0)), (name, k, t)
            if k == keys[-1]:
                for f in ('dyn', 'stat', 'meta', 'cnt', 'envi'):
                    a, b = getattr(st_m, f), getattr(twin.engine.state, f)
                    assert torch.equal(a.nan_to_num(-9.0) if a.is_floating_point() else a,
                                       b.nan_to_num(-9.0) if b.is_floating_point() else b), (name, f, t)
        firsts += int((ts_m.step_type == 0).sum())
    assert firsts > N, 'auto-resets happen during the run'
    # observation() draws every view again from the state
    obs = multi.observation()
    for k in keys:
        assert torch.equal(obs[k], twins[k][0].observation()[k]), k


@pytest.mark.gpu
def test_public_api_and_transports():
    """spawn_zoo with a RawState observer and a second renderer: step_to_host ('mapped', 'device',
    'chunked') and HostPipeline(depth=2) ('mapped', 'device') deliver the TimeSteps of step() plus
    explicit copies; VectorGymWrapper lists every image key with its own shape."""
    import torch
    from moog import observers
    from moog_b200.env_wrappers import VectorGymWrapper
    mod, cfg = _config('spawn_zoo')
    obs_cfg = dict(cfg['observers'], state=observers.RawState(),
                   side=_renderer(image_size=(128, 128), color_to_rgb='hsv_to_rgb'),
                   odd=_renderer(image_size=(7, 5), color_to_rgb='hsv_to_rgb'))   # 105-byte frames
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(6)]
    N, T = 192, 70    # the 60-step timeout: every env resets on the way
    keys = ('image', 'side', 'odd', 'state')
    env, _ = _env(cfg, mod, N, 21, states, obs_cfg, start=False)
    ts = env.reset()
    acts = _actions(env, T)
    ref = [{k: v.cpu().clone() for k, v in ts.observation.items()}]
    meta = [(ts.step_type.cpu().clone(), ts.reward.cpu().clone())]
    for a in acts:
        ts = env.step(a)
        assert set(ts.observation) == set(keys)
        assert ts.observation['side'] is env.engine.view_frames[0]
        ref.append({k: v.cpu().clone() for k, v in ts.observation.items()})
        meta.append((ts.step_type.cpu().clone(), ts.reward.cpu().clone()))

    def same(got, k, what):
        for key in keys:
            assert torch.equal(got.observation[key].cpu(), ref[k][key]), (what, key, k)
        assert torch.equal(got.step_type.cpu(), meta[k][0]), (what, k)
        assert torch.equal(got.reward.cpu().nan_to_num(-7.0), meta[k][1].nan_to_num(-7.0)), (what, k)

    pin = lambda t: torch.empty(t.shape, dtype=t.dtype).pin_memory()
    for mode in ('mapped', 'device', 'chunked'):
        twin, _ = _env(cfg, mod, N, 21, states, obs_cfg, start=False)   # the first call is the reset
        e = twin.engine
        host = type(ts)(pin(e.step_type), pin(e.reward), pin(e.discount),
                        {'image': pin(e.frames), 'side': pin(e.view_frames[0]), 'odd': pin(e.view_frames[1]),
                         'state': pin(e.sprites)})
        same(twin.step_to_host(None, host, frames=mode), 0, mode)
        for k, a in enumerate(acts, 1):
            same(twin.step_to_host(a, host, frames=mode), k, mode)
    for mode in ('mapped', 'device'):
        twin, _ = _env(cfg, mod, N, 21, states, obs_cfg, start=False)
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
    spaces = VectorGymWrapper(env).observation_space
    assert spaces['image']['shape'] == (64, 64, 3) and spaces['side']['shape'] == (128, 128, 3)
    assert spaces['odd']['shape'] == (5, 7, 3) and spaces['side']['dtype'] == 'uint8'
    assert spaces['state']['shape'] == (env.program.n_slots, 16)


def _clone(ts):
    return type(ts)(ts.step_type.clone(), ts.reward.clone(), ts.discount.clone(),
                    {k: v.clone() for k, v in ts.observation.items()})


@pytest.mark.gpu
@pytest.mark.parametrize('n_envs', [4096, 1001])
def test_views_at_size(n_envs):
    """4096 falling_balls20 envs (view 0 drawn by the tail render behind the step) and a batch that is
    not a multiple of the render kernel's envs per CTA, with a second 128 x 128 view: view 0 equals
    moog_render of the state the step left, view 1 what a program with only that renderer draws."""
    import torch
    from moog_b200 import compiler as C
    from moog_b200.batched_env import Engine
    mod, cfg = _config('falling_balls20', side=_renderer(image_size=(128, 128), bg_color=(5, 6, 7)))
    np.random.seed(9)
    states = [cfg['state_initializer']() for _ in range(64)]
    from moog_b200.batched_env import BatchedEnvironment
    env = BatchedEnvironment(**cfg, num_envs=n_envs, device='cuda:0', seed=2, initial_states=states)
    env.reset()
    rng = np.random.RandomState(1)
    for _ in range(3):
        ts = env.step(torch.from_numpy(rng.randint(0, 5, size=(n_envs, 1)).astype(np.float64)))
    e = env.engine
    if n_envs == 4096:
        assert not e.dev_program.step_draws_frames(n_envs)    # the render kernel, behind the step
    again = e.render(out=torch.zeros_like(e.frames))
    assert torch.equal(ts.observation['image'], again)
    alone = C.compile_config(dict(cfg, observers={'side': cfg['observers']['side']}), states)
    twin = Engine(alone, n_envs, 'cuda:0')
    twin.state.copy_from(e.state)
    assert torch.equal(ts.observation['side'], twin.render())


@pytest.mark.gpu
def test_nothing_else_changes():
    """V renderers launch exactly V - 1 more kernels per step than the program with view 0 alone; view
    0, state and rewards are bit-identical; a single-renderer step() launches what env_step does."""
    import torch
    from moog_b200 import capi
    mod, cfg = _config('spawn_zoo')
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(6)]
    N = 256
    extra = dict(a=_renderer(image_size=(32, 32)), b=_renderer(image_size=(64, 64), anti_aliasing=2),
                 c=_renderer(image_size=(256, 256), color_to_rgb='hsv_to_rgb'))
    one, _ = _env(cfg, mod, N, 3, states, cfg['observers'])
    many, _ = _env(cfg, mod, N, 3, states, dict(cfg['observers'], **extra))
    assert one.engine.view_frames == [] and one.engine.n_views == 1
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
        assert torch.equal(one.engine.state.dyn.nan_to_num(-9.0), many.engine.state.dyn.nan_to_num(-9.0)), k
    act = torch.from_numpy(_actions(one, 1, seed=8)[0])
    c0 = capi.launch_count()
    one.engine.env_step(act, frames=True)
    c1 = capi.launch_count()
    one.step(act)
    c2 = capi.launch_count()
    assert c2 - c1 == c1 - c0
