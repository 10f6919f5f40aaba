"""SpriteMask: which sprite each pixel shows, drawn by the frames' own scan conversion.

The oracle is Pillow itself, as in test_render_aa_large.pillow_render: a black RGB canvas,
ImageDraw.Draw(canvas, 'RGBA').polygon per live sprite with a non-zero ink alpha in slot order, with the
opaque ink ((s+1) & 255, (s+1) >> 8, 0, 255) -- opaque ink overwrites, so what it covers is what the
frames' fill covers -- decoded as R + 256 G - 1 and flipped.

Without a GPU: the program format, the compiler, validation, the plan, and the oracle against
Oracle.render.  On the GPU: moog_render_mask and every BatchedEnvironment path against the oracle,
0 differing pixels.
"""
import colorsys
import ctypes
import importlib
import os
import re

import numpy as np
import pytest

from tests import util

SIZES = [(64, 64), (84, 84), (136, 200), (256, 256)]   # (width, height), SpriteMask(image_size=...) order
HUGE = (1024, 1024)


def _config(name, **observers):
    import moog_b200  # noqa: F401
    mod = importlib.import_module('moog_b200.configs.' + name)
    cfg = mod.get_config()
    if observers:
        cfg['observers'] = dict(cfg['observers'], **observers)
    return mod, cfg


def _mask(**kw):
    from moog import observers
    return observers.SpriteMask(**kw)


def _split(blob):
    """(header, ops bytes, ipool, expr + dpool bytes) of a program blob."""
    from moog_b200 import compiler as C
    b = bytes(bytearray(blob))
    hdr = np.frombuffer(b[:C.HDR_WORDS * 4], dtype='<i4').copy()
    start = C.HDR_WORDS * 4 + 80 * int(hdr[C.H_N_OPS])
    n_ipool = int(hdr[C.H_N_IPOOL])
    ipool = np.frombuffer(b[start:start + 4 * n_ipool], dtype='<i4').copy()
    return hdr, b[C.HDR_WORDS * 4:start], ipool, b[start + 4 * ((n_ipool + 1) & ~1):]


def with_masks(blob, rows, table=None):
    """`blob` with a mask table of `rows` (lists of MOOG_VIEW_WORDS ints) appended to its ipool -- the
    layout compiler.Program.finalize writes for a config with len(rows) SpriteMasks.  `table`: the
    header's MOOG_H_MASKS instead of where the rows went."""
    from moog_b200 import compiler as C
    hdr, ops, ipool, rest = _split(blob)
    ipool = list(ipool)
    hdr[C.H_MASKS] = (len(ipool) if rows else 0) if table is None else table
    hdr[C.H_N_MASKS] = len(rows)
    ipool += [int(w) for r in rows for w in r]
    hdr[C.H_N_IPOOL] = len(ipool)
    if len(ipool) % 2:
        ipool.append(0)
    out = ops + np.asarray(ipool, dtype='<i4').tobytes() + rest
    hdr[C.H_BYTES] = C.HDR_WORDS * 4 + len(out)
    return hdr.tobytes() + out


def mask_row(width, height, modifier=0, mod_layer=0):
    return [height, width, 1, 0, 0, modifier, mod_layer, 1]


def _validate(blob):
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    buf = (ctypes.c_uint8 * len(blob)).from_buffer_copy(bytes(blob))
    return capi.lib().moog_program_validate(ctypes.cast(buf, ctypes.c_void_p), len(blob))


def _mask_plan(blob, k=0):
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    return capi.mask_plan(blob, k)


def _states(g, steps):
    parts = [util.state_at(g, int(t)) for t in steps]
    return {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}


def _steps(g, k=3):
    T = len(g['reward'])
    return [-1] + [int(t) for t in np.linspace(0, T - 1, k - 1).round()]


def _modifier(prog):
    """(modifier, agent layer) of the program's view 0."""
    from moog_b200 import compiler as C
    return int(prog.header[C.H_R_MODIFIER]), int(prog.header[C.H_R_MOD_LAYER])


def pillow_mask(prog, arrays, width, height, modifier=0, mod_layer=0):
    """SpriteMask on Pillow itself: int16 [n, height, width] (see the module docstring)."""
    from PIL import Image, ImageDraw
    from moog_b200 import compiler as C
    from oracle.oracle import Oracle
    verts, nv = Oracle(prog, arrays).world_vertices()
    out = []
    for n in range(arrays['dyn'].shape[0]):
        canvas = Image.new('RGB', (width, height), (0, 0, 0))
        draw = ImageDraw.Draw(canvas, 'RGBA')
        dyn, stat = arrays['dyn'][n], arrays['stat'][n]
        if modifier == C.PMOD_TORUS:     # polygon_modifiers.py TorusGeometry: 9 shifted copies
            shifts = [(float(c // 3 - 1), float(c % 3 - 1)) for c in range(9)]
        elif modifier == C.PMOD_FIRST_PERSON:   # the agent (first slot of its layer) at the centre
            a = prog.layer_off[mod_layer]
            shifts = [(0.5 - float(dyn[0, a]), 0.5 - float(dyn[1, a]))]
        else:
            shifts = [None]
        for l in range(prog.n_layers):
            for i in range(int(arrays['cnt'][n, l])):
                s = prog.layer_off[l] + i
                if int(stat[9, s]) & 255 == 0:           # ink alpha uint8(int64(opacity)) == 0: not drawn
                    continue
                fill = ((s + 1) & 255, (s + 1) >> 8, 0, 255)
                for sh in shifts:
                    v = verts[n, s, :nv[n, s]]
                    if sh is not None:
                        v = v + np.array(sh)
                    pts = v * np.array([width, height])
                    if len(pts):
                        draw.polygon([tuple(p) for p in pts], fill=fill)
        px = np.asarray(canvas).astype(np.int32)
        out.append(np.flipud(px[..., 0] + 256 * px[..., 1] - 1).astype(np.int16))
    return np.stack(out)


# ---------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------

def test_mask_words_match_the_header():
    from moog_b200 import compiler as C
    with open(os.path.join(util.ROOT, 'include', 'moog_b200_program.h')) as f:
        text = f.read()
    assert (C.H_MASKS, C.H_N_MASKS) == tuple(int(v) for v in re.search(
        r'MOOG_H_MASKS = (\d+),.*?MOOG_H_N_MASKS = (\d+),', text, re.S).groups()) == (62, 63)
    # the words were free before: no stored program uses them
    for name in util.SCENES:
        hdr = np.frombuffer(bytes(bytearray(util.load_golden(name)['blob']))[:C.HDR_WORDS * 4], dtype='<i4')
        assert hdr[C.H_MASKS] == 0 and hdr[C.H_N_MASKS] == 0, name


def test_compiler_keeps_mask_order():
    from moog import observers
    from moog_b200 import compiler as C
    from moog.observers import polygon_modifiers
    _, cfg = _config('timed_center')
    np.random.seed(2)
    states = [cfg['state_initializer']()]
    obs = dict(m1=_mask(image_size=(32, 16)), image=cfg['observers']['image'], state=observers.RawState(),
               m0=_mask(image_size=(64, 64), polygon_modifier=polygon_modifiers.TorusGeometry(['agent'])),
               side=observers.PILRenderer(image_size=(48, 48)),
               fp=_mask(image_size=(75, 75), polygon_modifier=cfg['observers']['image'].polygon_modifier))
    prog = C.compile_config(dict(cfg, observers=obs), states)
    assert [k for k, _ in prog.masks] == ['m1', 'm0', 'fp']
    assert [k for k, _ in prog.views] == ['image', 'side'] and prog.state_key == 'state'
    hdr, _, ipool, _ = _split(prog.blob)
    assert hdr[C.H_N_MASKS] == 3 and hdr[C.H_N_VIEWS] == 1
    table = ipool[hdr[C.H_MASKS]:hdr[C.H_MASKS] + 3 * C.VIEW_WORDS].reshape(3, C.VIEW_WORDS).tolist()
    agent = prog.layer_index('agent')
    assert table == [mask_row(32, 16), mask_row(64, 64, C.PMOD_TORUS),
                     mask_row(75, 75, C.PMOD_FIRST_PERSON, agent)]
    assert _validate(prog.blob) == 0
    # without the masks: the same program, word for word, up to the table
    plain = C.compile_config(dict(cfg, observers={k: v for k, v in obs.items() if k[0] != 'm' and k != 'fp'}), states)
    h0, ops0, ip0, rest0 = _split(plain.blob)
    h1, ops1, ip1, rest1 = _split(prog.blob)
    assert ops0 == ops1 and rest0 == rest1 and np.array_equal(ip1[:len(ip0)], ip0)
    assert hdr[C.H_MASKS] == len(ip0) and len(ip1) == len(ip0) + 3 * C.VIEW_WORDS
    diff = sorted(int(w) for w in np.nonzero(h0 != h1)[0])
    assert diff == sorted([C.H_BYTES, C.H_N_IPOOL, C.H_MASKS, C.H_N_MASKS]), diff
    # and with every mask removed by hand, the same bytes
    assert with_masks(plain.blob, []) == plain.blob


def test_mask_without_a_renderer_and_the_ninth_mask():
    from moog_b200 import compiler as C
    _, cfg = _config('falling_balls20')
    np.random.seed(2)
    states = [cfg['state_initializer']()]
    prog = C.compile_config(dict(cfg, observers={'mask': _mask(image_size=(40, 30))}), states)
    assert prog.render is None and prog.views == [] and [k for k, _ in prog.masks] == ['mask']
    assert prog.masks[0][1]['width'] == 40 and prog.masks[0][1]['height'] == 30
    assert _validate(prog.blob) == 0
    assert _mask_plan(prog.blob)[0] == 0
    eight = {'m%d' % k: _mask(image_size=(16, 16)) for k in range(8)}
    assert len(C.compile_config(dict(cfg, observers=eight), states).masks) == 8
    with pytest.raises(C.CompileError, match='at most 8 SpriteMask'):
        C.compile_config(dict(cfg, observers=dict(eight, m8=_mask())), states)


def test_mask_table_is_validated():
    from moog_b200 import compiler as C
    g = util.load_golden('timed_center')
    blob = g['blob'].tobytes()
    L = g['program'].n_layers
    good = [mask_row(64, 64), mask_row(7, 5, C.PMOD_TORUS), mask_row(8192, 1, C.PMOD_FIRST_PERSON, L - 1)]
    assert _validate(with_masks(blob, good)) == 0
    assert _validate(with_masks(blob, [mask_row(16, 16)] * 8)) == 0

    def bad_row(word, value):
        rows = [list(r) for r in good]
        rows[1][word] = value
        return with_masks(blob, rows)
    for word, value in [(2, 2), (2, 0), (0, 0), (1, 0), (0, -3), (1, 8193), (3, 1), (4, 1), (5, 3), (5, -1),
                        (7, 0), (7, 2)]:
        assert _validate(bad_row(word, value)) == -1, (word, value)
    rows = [list(r) for r in good]
    rows[2][6] = L            # the agent layer out of range
    assert _validate(with_masks(blob, rows)) == -1
    assert _validate(with_masks(blob, [mask_row(16, 16)] * 9)) == -1
    n_ipool = int(_split(blob)[0][C.H_N_IPOOL])
    assert _validate(with_masks(blob, good, table=n_ipool + 1)) == -1      # the table runs past the pool
    assert _validate(with_masks(blob, good, table=-1)) == -1
    hdr, ops, ipool, rest = _split(with_masks(blob, good))
    hdr[C.H_N_MASKS] = -1
    assert _validate(hdr.tobytes() + bytes(bytearray(with_masks(blob, good)))[C.HDR_WORDS * 4:]) == -1


def test_mask_plan_covers_every_size_up_to_1024():
    import moog_b200  # noqa: F401
    from moog_b200 import capi, compiler as C
    sides = [1, 7, 16, 50, 64, 75, 84, 128, 136, 200, 256, 333, 512, 777, 1000, 1024]
    for scene in util.AA_SCENES:
        blob = util.load_golden(scene)['blob'].tobytes()
        for w in sides:
            blobs = with_masks(blob, [mask_row(w, h) for h in sides[:8]])
            for k in range(8):
                code, rows, smem = _mask_plan(blobs, k)
                assert code == 0 and 1 <= rows <= sides[k] and 0 < smem <= 224 * 1024, (scene, w, sides[k])
            blobs = with_masks(blob, [mask_row(w, h) for h in sides[8:]])
            for k in range(len(sides) - 8):
                code, rows, smem = _mask_plan(blobs, k)
                assert code == 0 and 1 <= rows <= sides[8 + k] and 0 < smem <= 224 * 1024, (scene, w, sides[8 + k])
    # TorusGeometry: 9 copies of cleanup's outlines do not fit a CTA next to any band
    blob = util.load_golden('cleanup')['blob'].tobytes()
    assert _mask_plan(with_masks(blob, [mask_row(64, 64, C.PMOD_TORUS)]))[0] == capi.E_UNSUPPORTED
    code = _mask_plan(with_masks(util.load_golden('chase_avoid_torus')['blob'].tobytes(),
                                 [mask_row(256, 256, C.PMOD_TORUS)]))[0]
    assert code == 0
    for bad in (-1, 1):
        assert _mask_plan(with_masks(blob, [mask_row(64, 64)]), bad)[0] == capi.E_INVAL
    assert _mask_plan(blob, 0)[0] == capi.E_INVAL        # no mask table
    assert capi.lib().moog_mask_plan(None, 0, 0, None, None) == capi.E_INVAL


def test_undrawable_mask_is_named_before_anything_runs():
    from moog_b200 import capi, compiler as C
    from moog_b200.batched_env import Engine
    from moog.observers import polygon_modifiers
    _, cfg = _config('cleanup64')
    np.random.seed(3)
    states = [cfg['state_initializer']()]
    torus = polygon_modifiers.TorusGeometry(list(states[0].keys()))
    prog = C.compile_config(dict(cfg, observers=dict(cfg['observers'], who=_mask(polygon_modifier=torus))), states)
    with pytest.raises(capi.MoogError, match=r"'who'.*SpriteMask\(image_size=\(64, 64\)\)"):
        Engine._check_views(prog)
    Engine._check_views(C.compile_config(dict(cfg, observers=dict(cfg['observers'], who=_mask(image_size=(1024, 1024)))),
                                         states))


def _inks(prog, arrays, cmap):
    """[n, S, 3] uint8 RGB ink of every slot, as the frames compute it."""
    from moog_b200 import compiler as C
    u8 = lambda v: int(v) & 255
    n, S = arrays['stat'].shape[0], prog.n_slots
    out = np.zeros((n, S, 3), dtype=np.uint8)
    for e in range(n):
        for s in range(S):
            c = [float(arrays['stat'][e, k, s]) for k in (6, 7, 8)]
            if cmap == C.CMAP_HSV:
                c = [255 * v for v in colorsys.hsv_to_rgb(*c)]
            out[e, s] = [u8(v) for v in c]
    return out


def test_oracle_mask_colours_into_the_frames():
    """On golden states whose drawn sprites are all opaque, the Pillow mask coloured with each slot's ink
    (the background where -1) is Oracle.render at anti_aliasing 1, byte for byte."""
    from moog_b200 import compiler as C
    from oracle.oracle import Oracle
    checked = []
    for scene in util.SCENES:
        g = util.load_golden(scene)
        prog = g['program']
        hdr = prog.header
        H, W, aa, bg, cmap = (int(v) for v in hdr[C.H_R_HEIGHT:C.H_R_COLORMAP + 1])
        if not hdr[C.H_R_ENABLED] or aa != 1:
            continue
        steps = [t for t in _steps(g, 4)
                 if all(int(v) & 255 in (0, 255) for v in _opacities(prog, util.state_at(g, t)))]
        if not steps:
            continue
        arrays = _states(g, steps)
        mask = pillow_mask(prog, arrays, W, H, *_modifier(prog))
        ink = _inks(prog, arrays, cmap)
        bgc = np.array([bg & 255, (bg >> 8) & 255, (bg >> 16) & 255], dtype=np.uint8)
        want = Oracle(prog, arrays).render()
        got = np.where((mask >= 0)[..., None], ink[np.arange(len(steps))[:, None, None], np.maximum(mask, 0)], bgc)
        assert int((got != want).sum()) == 0, scene
        checked.append(scene)
    assert len(checked) >= 8, checked


def _opacities(prog, st):
    live = util.live_mask(prog, st['cnt'][0])
    return st['stat'][0, 9, live]


# ---------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------

def _masked_stub(g, sizes, modifier=0, mod_layer=0):
    prog = util.ProgramStub(with_masks(g['blob'].tobytes(), [mask_row(w, h, modifier, mod_layer) for w, h in sizes]),
                            g['layer_names'])
    prog.masks = [('m%d' % k, dict(width=w, height=h)) for k, (w, h) in enumerate(sizes)]
    return prog


@pytest.mark.gpu
@pytest.mark.parametrize('scene', util.SCENES)
def test_mask_kernel_matches_pillow(scene):
    """moog_render_mask at 64 x 64, 84 x 84, 136 x 200 and 256 x 256 on states across the golden
    trajectory, and at 1024 x 1024 (bands) on one, with the scene's polygon modifier (FirstPersonAgent
    in timed_center, TorusGeometry in chase_avoid_torus): 0 differing pixels against Pillow."""
    import torch
    from moog_b200.batched_env import Engine
    g = util.load_golden(scene)
    mod = _modifier(g['program'])
    prog = _masked_stub(g, SIZES + [HUGE], *mod)
    arrays = _states(g, _steps(g))
    eng = Engine(prog, arrays['dyn'].shape[0], 'cuda:0')
    eng.state.upload(arrays)
    for k, (w, h) in enumerate(SIZES + [HUGE]):
        sub = arrays if (w, h) != HUGE else {key: v[:1] for key, v in arrays.items()}
        got = eng.render_mask(mask=k).cpu().numpy()[:sub['dyn'].shape[0]]
        want = pillow_mask(g['program'], sub, w, h, *mod)
        assert got.shape == want.shape == (sub['dyn'].shape[0], h, w)
        assert int((got != want).sum()) == 0, (scene, w, h)
    # a range, into pinned host memory
    host = torch.full(eng.masks[2].shape, 7, dtype=torch.int16).pin_memory()
    eng.render_mask(out=host, first=1, count=eng.n - 1, mask=2)
    torch.cuda.synchronize()
    assert torch.equal(host[1:], eng.masks[2][1:].cpu()) and bool((host[0] == 7).all())


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


ENV_AGE = {'falling_balls20': 0, 'spawn_zoo': 0, 'colliding_predators84': 150}


@pytest.mark.gpu
@pytest.mark.parametrize('name, reset_mode', [('falling_balls20', 'pool'), ('spawn_zoo', 'pool'),
                                              ('colliding_predators84', 'device')])
def test_environment_masks_match_pillow(name, reset_mode):
    """A BatchedEnvironment with two SpriteMasks stepped 100 times through auto-resets: every step's masks
    equal Pillow's on the downloaded state, every slot they name is live in that step's RawState, and the
    frames equal those of a twin without masks."""
    import torch
    from moog import observers
    mod, cfg = _config(name)
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(6)]
    N, T = 12, 100
    obs = dict(cfg['observers'], state=observers.RawState(), mask=_mask(image_size=(64, 64)),
               odd=_mask(image_size=(75, 50)))
    env, ts = _env(cfg, mod, N, 7, states, obs, reset_mode, ENV_AGE[name])
    twin, ts_t = _env(cfg, mod, N, 7, states, cfg['observers'], reset_mode, ENV_AGE[name])
    prog = env.program
    acts = _actions(env, T)
    firsts = 0
    for t in range(T + 1):
        if t > 0:
            ts, ts_t = env.step(acts[t - 1]), twin.step(acts[t - 1])
        assert torch.equal(ts.observation['image'], ts_t.observation['image']), (name, t)
        arrays = env.engine.state.download()
        alive = ts.observation['state'][..., 15].cpu().numpy() > 0
        for k, key in enumerate(('mask', 'odd')):
            m = prog.masks[k][1]
            got = ts.observation[key].cpu().numpy()
            want = pillow_mask(prog, arrays, m['width'], m['height'])
            assert int((got != want).sum()) == 0, (name, key, t)
            e, s = np.nonzero(got >= 0)[0], got[got >= 0]
            assert alive[e, s].all(), (name, key, t)
        firsts += int((ts.step_type == 0).sum())
    assert firsts > N, 'auto-resets happen during the run'
    obs_again = env.observation()
    assert torch.equal(obs_again['mask'], ts.observation['mask'])


def _clone(ts):
    return type(ts)(ts.step_type.clone(), ts.reward.clone(), ts.discount.clone(),
                    {k: v.clone() for k, v in ts.observation.items()})


@pytest.mark.gpu
@pytest.mark.parametrize('n_envs', [4096, 1001])
def test_masks_through_every_transport(n_envs):
    """falling_balls20 with a 64 x 64 and a 75 x 75 mask (11250 bytes per env: drawn whole under 'chunked')
    and a RawState: step_to_host ('mapped', 'device', 'chunked') and HostPipeline(depth=2) ('mapped',
    'device') deliver what step() returns; VectorGymWrapper lists the masks."""
    import torch
    from moog import observers
    from moog_b200.env_wrappers import VectorGymWrapper
    mod, cfg = _config('falling_balls20')
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(16)]
    obs = dict(cfg['observers'], state=observers.RawState(), mask=_mask(image_size=(64, 64)),
               odd=_mask(image_size=(75, 75)))
    keys = ('image', 'state', 'mask', 'odd')
    T = 12
    env, _ = _env(cfg, mod, n_envs, 21, states, obs, start=False)
    ts = env.reset()
    acts = _actions(env, T)
    ref = [{k: v.cpu().clone() for k, v in ts.observation.items()}]
    meta = [(ts.step_type.cpu().clone(), ts.reward.cpu().clone())]
    for a in acts:
        ts = env.step(a)
        assert set(ts.observation) == set(keys)
        assert ts.observation['mask'] is env.engine.masks[0]
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
                        {'image': pin(e.frames), 'state': pin(e.sprites), 'mask': pin(e.masks[0]),
                         'odd': pin(e.masks[1])})
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
    spaces = VectorGymWrapper(env).observation_space
    S = env.program.n_slots
    assert spaces['mask'] == dict(low=-1, high=S - 1, shape=(64, 64), dtype='int16')
    assert spaces['odd']['shape'] == (75, 75)


@pytest.mark.gpu
def test_launches_and_frames_with_masks():
    """M masks launch exactly M more kernels per step; frames, state and rewards are those of the program
    without masks; a program without a mask launches what env_step does."""
    import torch
    from moog_b200 import capi
    mod, cfg = _config('spawn_zoo')
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(6)]
    N = 256
    extra = dict(a=_mask(image_size=(32, 32)), b=_mask(image_size=(256, 256)), c=_mask(image_size=(75, 75)))
    one, _ = _env(cfg, mod, N, 3, states, cfg['observers'])
    many, _ = _env(cfg, mod, N, 3, states, dict(cfg['observers'], **extra))
    assert one.engine.masks == [] and len(many.engine.masks) == 3
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
    act = torch.from_numpy(_actions(one, 1, seed=8)[0])
    c0 = capi.launch_count()
    one.engine.env_step(act, frames=True)
    c1 = capi.launch_count()
    one.step(act)
    c2 = capi.launch_count()
    assert c2 - c1 == c1 - c0


@pytest.mark.gpu
def test_undrawable_mask_is_refused_at_construction():
    from moog_b200 import capi
    from moog_b200.batched_env import BatchedEnvironment
    from moog.observers import polygon_modifiers
    mod, cfg = _config('cleanup64')
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(2)]
    torus = polygon_modifiers.TorusGeometry(list(states[0].keys()))
    with pytest.raises(capi.MoogError, match=r"observer 'who'"):
        BatchedEnvironment(**dict(cfg, observers=dict(cfg['observers'], who=_mask(polygon_modifier=torus))),
                           num_envs=4, device='cuda:0', initial_states=states,
                           layer_capacity=getattr(mod, 'LAYER_CAPACITY', None))
