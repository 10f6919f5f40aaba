"""Anti-aliased frames at every image size up to 1024 x 1024.

PILRenderer(anti_aliasing=k) draws on a canvas k times the image size and resizes it with Pillow's
LANCZOS filter (pil_renderer.py:88-120).  The render kernel draws such a canvas in chunks of rows and
streams every chunk through the resize (moog_render_dev.cuh render_env_aa), so the canvas never has
to fit one CTA's shared memory whole.  `moog_render_plan` says how a view is drawn, or that it cannot
be, and BatchedEnvironment refuses such a view when it is built.

Without a GPU: Oracle.render (the C restatement of PILRenderer) against Pillow itself at the new
sizes, and the plan's coverage.  On the GPU: every frame path against Oracle.render, 0 differing
bytes.
"""
import colorsys
import ctypes
import importlib

import numpy as np
import pytest

from tests import util

# (width, height, anti_aliasing), PILRenderer(image_size=(width, height)) order
SIZES = [(84, 84, 3), (128, 128, 2), (256, 256, 2), (64, 64, 4), (136, 200, 3)]
HUGE = (1024, 1024, 2)   # one state per scene


def _program(g, width, height, aa, modifier=None):
    """The golden scene's program with view 0 = PILRenderer(image_size=(width, height), anti_aliasing=aa)."""
    from moog_b200 import compiler as C
    prog = util.with_image_size(g, width, height)
    blob = np.frombuffer(prog.blob, dtype=np.uint8).copy()
    hdr = blob[:C.HDR_WORDS * 4].view('<i4')
    hdr[C.H_R_AA] = aa
    if modifier is not None:
        hdr[C.H_R_MODIFIER] = modifier
    return util.ProgramStub(blob, g['layer_names'])


def _states(g, steps):
    parts = [util.state_at(g, int(t)) for t in steps]
    return {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}


def _steps(g, k=3):
    T = len(g['reward'])
    return [-1] + [int(t) for t in np.linspace(0, T - 1, k - 1).round()]


def _plan(blob, view=0):
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    return capi.render_plan(blob, view)


# ---------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------

def pillow_render(prog, arrays):
    """PILRenderer.__call__ on Pillow itself (SURVEY App. B.8): background; ImageDraw.Draw(canvas,
    'RGBA').polygon per live sprite in z-order, vertices = world vertices x the canvas size; colours
    through hsv_to_rgb where the scene uses it; resize(image_size, LANCZOS); flipud."""
    from PIL import Image, ImageDraw
    from moog_b200 import compiler as C
    from oracle.oracle import Oracle
    hdr = prog.header
    H, W, aa, bg, cmap, pmod = (int(v) for v in hdr[C.H_R_HEIGHT:C.H_R_MODIFIER + 1])
    assert pmod == C.PMOD_NONE
    verts, nv = Oracle(prog, arrays).world_vertices()
    u8 = lambda v: int(v) & 255   # (uint8)(long long)v, color_maps.py / Pillow's ink
    frames = []
    for n in range(arrays['dyn'].shape[0]):
        canvas = Image.new('RGB', (aa * W, aa * H), (bg & 255, (bg >> 8) & 255, (bg >> 16) & 255))
        draw = ImageDraw.Draw(canvas, 'RGBA')
        stat = arrays['stat'][n]
        for l in range(prog.n_layers):
            for i in range(int(arrays['cnt'][n, l])):
                s = prog.layer_off[l] + i
                c = [float(stat[k, s]) for k in (6, 7, 8)]          # MOOG_S_C0 .. C2
                if cmap == C.CMAP_HSV:
                    c = [255 * v for v in colorsys.hsv_to_rgb(*c)]
                fill = tuple(u8(v) for v in c) + (u8(stat[9, s]),)  # MOOG_S_OPACITY
                pts = verts[n, s, :nv[n, s]] * np.array([aa * W, aa * H])
                if len(pts):
                    draw.polygon([tuple(p) for p in pts], fill=fill)
        frames.append(np.flipud(np.asarray(canvas.resize((W, H), Image.LANCZOS))))
    return np.stack(frames)


def test_stat_columns_match_the_header():
    import os
    import re
    with open(os.path.join(util.ROOT, 'include', 'moog_b200_program.h')) as f:
        text = f.read()
    enum = re.search(r'enum \{\s*(MOOG_S_MASS = 0,[^}]*)\}', text).group(1)
    names = [n.split('=')[0].strip() for n in enum.split(',')]
    assert [names.index('MOOG_S_' + k) for k in ('C0', 'C1', 'C2', 'OPACITY')] == [6, 7, 8, 9]


@pytest.mark.parametrize('scene', util.AA_SCENES)
def test_oracle_matches_pillow_at_new_sizes(scene):
    """Oracle.render == Pillow's PILRenderer on golden states at the sizes no recording covers."""
    from oracle.oracle import Oracle
    g = util.load_golden(scene)
    for w, h, aa in SIZES + [HUGE]:
        steps = _steps(g)[:1] if (w, h, aa) == HUGE else _steps(g)
        prog = _program(g, w, h, aa)
        arrays = _states(g, steps)
        got = Oracle(prog, arrays).render()
        want = pillow_render(prog, arrays)
        assert got.shape == want.shape == (len(steps), h, w, 3)
        assert int((got != want).sum()) == 0, (scene, w, h, aa)


def test_plan_covers_every_image_up_to_1024():
    """Every image up to 1024 x 1024 (square or not) at anti_aliasing 2, 3, 4 for the AA_SCENES
    programs, and TorusGeometry up to 256 x 256 at anti_aliasing 2: accepted, <= 224 KB per env."""
    from moog_b200 import compiler as C
    sides = [1, 7, 16, 50, 64, 75, 84, 97, 128, 136, 200, 256, 333, 512, 640, 777, 1000, 1024]
    for scene in util.AA_SCENES:
        g = util.load_golden(scene)
        for aa in (2, 3, 4):
            for w in sides:
                for h in sides:
                    code, rows, smem = _plan(_program(g, w, h, aa).blob)
                    assert code == 0, (scene, w, h, aa)
                    assert 1 <= rows <= aa * h and 0 < smem <= 224 * 1024, (scene, w, h, aa, rows, smem)
    # TorusGeometry draws 9 copies of every outline: the edge lists of cleanup's 826 vertices alone
    # exceed a CTA's shared memory at any image size (anti_aliasing 1 included)
    for scene in ['pong', 'falling_balls20', 'colliding_predators', 'chase_avoid_torus']:
        g = util.load_golden(scene)
        for side in (64, 128, 200, 256):
            code, rows, smem = _plan(_program(g, side, side, 2, modifier=C.PMOD_TORUS).blob)
            assert code == 0 and smem <= 224 * 1024, (scene, side)
    g = util.load_golden('cleanup')
    assert _plan(_program(g, 64, 64, 1, modifier=C.PMOD_TORUS).blob)[0] == -4


def _band_before(prog, width, height):
    """The anti_aliasing 1 band (rows, shared-memory bytes per env) that launch_render chose before the
    plan existed: render_layout of the whole canvas, else the largest multiple of 8 rows within 110 KB
    (8 at least).  A restatement of that code, to pin that the plan keeps it."""
    S, VT = prog.n_slots, max(prog.n_vtx, 1)

    def total(rows):
        o = (4 * rows * (width + 1) + 7) & ~7
        o += 24 * VT + max(8 * VT, 16 * min(max(S * 8, 512), 2048)) + 4 * S * 5 + 4 * (S + 1)
        return (o + 15) & ~15
    band = 0
    if total(height) > 110 * 1024:
        band = height & ~7
        while band > 8 and total(band) > 110 * 1024:
            band -= 8
    rows = band if band > 0 else height
    return rows, total(rows)


def test_plan_anti_aliasing_1_bands():
    """anti_aliasing 1 keeps its bands: the whole canvas while it fits 110 KB, else the largest multiple
    of 8 rows that does (8 rows at least) -- the rows and bytes launch_render chose before."""
    for scene in util.AA_SCENES + ['pacman']:
        g = util.load_golden(scene)
        assert _plan(g['blob'].tobytes())[:2] == (0, 64), scene
        for w, h in [(64, 64), (128, 128), (256, 256), (512, 512), (136, 200), (1024, 1024), (4096, 64), (200, 777)]:
            prog = _program(g, w, h, 1)
            code, rows, smem = _plan(prog.blob)
            assert code == 0, (scene, w, h)
            assert (rows, smem) == _band_before(prog, w, h), (scene, w, h, rows, smem)


def test_plan_refuses_what_no_chunk_holds():
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    g = util.load_golden('pong')
    assert _plan(_program(g, 8192, 64, 1).blob)[0] == -4         # one canvas row alone is 96 KB ... 8192 x 4 B
    assert _plan(_program(g, 4096, 4096, 4).blob)[0] == -4
    assert _plan(_program(g, 8192, 8, 16).blob)[0] == -4
    blob = g['blob'].tobytes()
    for bad in (-1, 1, 8):
        assert _plan(blob, bad)[0] == -1
    L = capi.lib()
    assert L.moog_render_plan(None, 0, 0, None, None) == -1
    buf = ctypes.create_string_buffer(blob, len(blob))
    assert L.moog_render_plan(buf, len(blob) - 8, 0, None, None) == -1   # malformed
    assert L.moog_render_plan(buf, len(blob), 0, None, None) == 0        # NULL outputs are optional


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


def test_undrawable_view_is_named_before_anything_runs():
    """Engine refuses a view no chunk holds with the observer key, its image_size and anti_aliasing."""
    from moog_b200 import capi, compiler as C
    from moog_b200.batched_env import Engine
    _, cfg = _config('spawn_zoo', big=_renderer(image_size=(4096, 4096), anti_aliasing=4))
    np.random.seed(3)
    prog = C.compile_config(cfg, [cfg['state_initializer']()])
    with pytest.raises(capi.MoogError, match=r"'big'.*image_size=\(4096, 4096\), anti_aliasing=4"):
        Engine._check_views(prog)
    _, cfg = _config('spawn_zoo', video=_renderer(image_size=(1024, 1024), anti_aliasing=2))
    Engine._check_views(C.compile_config(cfg, [cfg['state_initializer']()]))


# ---------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------

def _engine(prog, arrays):
    from moog_b200.batched_env import Engine
    eng = Engine(prog, arrays['dyn'].shape[0], 'cuda:0')
    eng.state.upload(arrays)
    return eng


@pytest.mark.gpu
@pytest.mark.parametrize('scene', util.AA_SCENES)
def test_render_kernel_matches_oracle(scene):
    """moog_render over a tiled batch (37 envs: not a multiple of envs per CTA), a batch of 2, ranged
    renders and a pinned host destination: 0 differing bytes against Oracle.render."""
    import torch
    from oracle.oracle import Oracle
    g = util.load_golden(scene)
    for w, h, aa in SIZES + [HUGE, (75, 50, 3)]:
        steps = _steps(g)[:1] if (w, h, aa) == HUGE else _steps(g)
        prog = _program(g, w, h, aa)
        one = _states(g, steps)
        want1 = Oracle(prog, one).render()
        n = 37 if (w, h, aa) != HUGE else 5
        idx = np.arange(n) % len(steps)
        arrays = {k: v[idx] for k, v in one.items()}
        want = want1[idx]
        eng = _engine(prog, arrays)
        got = eng.render(out=torch.full_like(eng.frames, 7)).cpu().numpy()
        assert int((got != want).sum()) == 0, (scene, w, h, aa)
        small = _engine(prog, {k: v[:2] for k, v in arrays.items()})
        assert int((small.render().cpu().numpy() != want[:2]).sum()) == 0, (scene, w, h, aa, 'small')
        # ranges (the 'chunked' transport renders [first, first + count)); 75 x 50 frames are not a
        # multiple of 16 bytes
        out = torch.full_like(eng.frames, 7)
        cuts = [0, n // 3, n // 3 + n // 4, n]
        for first, last in zip(cuts[:-1], cuts[1:]):
            eng.render(out=out, first=first, count=last - first)
        assert int((out.cpu().numpy() != want).sum()) == 0, (scene, w, h, aa, 'ranges')
        pinned = torch.full(tuple(eng.frames.shape), 9, dtype=torch.uint8).pin_memory()
        eng.render(out=pinned)
        torch.cuda.synchronize()
        assert int((pinned.numpy() != want).sum()) == 0, (scene, w, h, aa, 'pinned')


def _oracle_frames(prog, arrays):
    """Oracle.render of every env, each distinct state drawn once."""
    from oracle.oracle import Oracle
    n = arrays['dyn'].shape[0]
    keys = [b''.join(np.ascontiguousarray(arrays[k][i]).tobytes() for k in util.STATE_KEYS) for i in range(n)]
    first = {}
    for i, key in enumerate(keys):
        first.setdefault(key, i)
    rows = sorted(set(first.values()))
    frames = Oracle(prog, {k: v[rows] for k, v in arrays.items()}).render()
    where = {r: j for j, r in enumerate(rows)}
    return frames[[where[first[key]] for key in keys]]


@pytest.mark.gpu
@pytest.mark.parametrize('n', [1024, 6])
@pytest.mark.parametrize('scene', util.AA_SCENES)
def test_step_call_frames(scene, n):
    """moog_env_step with frames at 1024 envs (the persistent render kernel behind the step) and at 6
    envs (the render kernel after it), at every listed size: the frames are the oracle's render of the
    state each env was left in."""
    import torch
    g = util.load_golden(scene)
    steps = _steps(g, 8)
    one = _states(g, steps)
    for w, h, aa in SIZES + [(75, 50, 3)]:
        prog = _program(g, w, h, aa)
        idx = np.arange(n) % len(steps)
        eng = _engine(prog, {k: v[idx] for k, v in one.items()})
        eng.env_step(np.zeros((n, max(prog.action_dim, 1))), auto_reset=False, frames=True)
        got = eng.frames.cpu().numpy()
        torch.cuda.synchronize()
        want = _oracle_frames(prog, eng.state.download())
        assert int((got != want).sum()) == 0, (scene, w, h, aa, n)


@pytest.mark.gpu
def test_view_1_beside_an_unaliased_view_0():
    """moog_render_view draws anti-aliased views 1.. (up to 1024 x 1024 at anti_aliasing 2) next to a
    64 x 64 anti_aliasing 1 view 0."""
    from moog_b200 import compiler as C
    from oracle.oracle import Oracle
    from tests.test_render_views import with_views
    for scene in util.AA_SCENES:
        g = util.load_golden(scene)
        hdr = np.frombuffer(g['blob'].tobytes()[:C.HDR_WORDS * 4], dtype='<i4')
        rows = []
        for w, h, aa in SIZES + [HUGE]:
            r = [int(v) for v in hdr[C.H_R_HEIGHT:C.H_R_ENABLED + 1]]
            r[:3] = [h, w, aa]
            rows.append(r)
        prog = util.ProgramStub(with_views(g['blob'], rows), g['layer_names'])
        prog.views = [('image', prog.render)] + [('v%d' % k, dict(height=r[0], width=r[1], aa=r[2]))
                                                 for k, r in enumerate(rows, 1)]
        arrays = _states(g, _steps(g))
        eng = _engine(prog, arrays)
        assert int((eng.render().cpu().numpy() != Oracle(g['program'], arrays).render()).sum()) == 0
        for v, (w, h, aa) in enumerate(SIZES + [HUGE], 1):
            want = Oracle(_program(g, w, h, aa), arrays).render()
            assert int((eng.render(view=v).cpu().numpy() != want).sum()) == 0, (scene, w, h, aa)


@pytest.mark.gpu
def test_torus_and_first_person_at_128_aa2():
    from oracle.oracle import Oracle
    for scene in ('chase_avoid_torus', 'timed_center'):   # TorusGeometry, FirstPersonAgent
        g = util.load_golden(scene)
        prog = _program(g, 128, 128, 2)
        arrays = _states(g, _steps(g, 6))
        got = _engine(prog, arrays).render().cpu().numpy()
        assert int((got != Oracle(prog, arrays).render()).sum()) == 0, scene


def _env(cfg, mod, N, seed, states, observers):
    import torch
    from moog_b200.batched_env import BatchedEnvironment
    env = BatchedEnvironment(**dict(cfg, observers=observers), num_envs=N, device='cuda:0', seed=seed,
                             initial_states=states, layer_capacity=getattr(mod, 'LAYER_CAPACITY', None))
    ts = env.reset()
    env.engine.state.envi[:, 0] = torch.from_numpy(np.random.RandomState(4).randint(0, 30, size=N)).to(
        'cuda:0', dtype=torch.int32)       # staggered time-outs: auto-resets at many steps
    return env, ts


@pytest.mark.gpu
def test_public_api_video_view():
    """BatchedEnvironment with {'image': 64 x 64, 'video': 256 x 256 anti_aliasing 2}: 50 steps with
    auto-resets, every step's 'video' is the oracle's render of the state; step_to_host ('mapped',
    'device', 'chunked') and HostPipeline deliver the same frames; one render launch per AA view; an
    undrawable view is refused at construction, naming its key."""
    import torch
    from moog_b200 import capi, compiler as C
    from oracle.oracle import Oracle
    mod, cfg = _config('spawn_zoo')
    video = _renderer(image_size=(256, 256), anti_aliasing=2, color_to_rgb='hsv_to_rgb')
    obs = dict(cfg['observers'], video=video)
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(6)]
    alone = C.compile_config(dict(cfg, observers={'video': video}), states,
                             layer_capacity=getattr(mod, 'LAYER_CAPACITY', None))
    N, T = 24, 50
    env, ts = _env(cfg, mod, N, 21, states, obs)
    one, _ = _env(cfg, mod, N, 21, states, cfg['observers'])
    rng = np.random.RandomState(5)
    acts = [rng.uniform(-1, 1, size=(N, env.action_dim)) for _ in range(T)]
    ref, firsts = [ts.observation['video'].cpu().clone()], 0
    for k, a in enumerate(acts):
        c0 = capi.launch_count()
        ts = env.step(a)
        c1 = capi.launch_count()
        one.step(a)
        c2 = capi.launch_count()
        assert (c1 - c0) - (c2 - c1) == 1, k
        want = Oracle(alone, env.engine.state.download()).render()
        assert int((ts.observation['video'].cpu().numpy() != want).sum()) == 0, k
        ref.append(ts.observation['video'].cpu().clone())
        firsts += int((ts.step_type == 0).sum())
    assert firsts > 0, 'auto-resets happen during the run'
    pin = lambda t: torch.empty(t.shape, dtype=t.dtype).pin_memory()
    for mode in ('mapped', 'device', 'chunked'):
        twin, _ = _env(cfg, mod, N, 21, states, obs)
        e = twin.engine
        host = type(ts)(pin(e.step_type), pin(e.reward), pin(e.discount),
                        {'image': pin(e.frames), 'video': pin(e.view_frames[0])})
        for k, a in enumerate(acts[:10], 1):
            got = twin.step_to_host(a, host, frames=mode)
            assert torch.equal(got.observation['video'].cpu(), ref[k]), (mode, k)
    for mode in ('mapped', 'device'):
        twin, _ = _env(cfg, mod, N, 21, states, obs)
        pipe = twin.host_pipeline(depth=2, frames=mode)
        got = []
        for k, a in enumerate(acts[:10]):
            if k >= 2:
                got.append(pipe.collect().observation['video'].cpu().clone())
            pipe.submit(a)
        while len(got) < 10:
            got.append(pipe.collect().observation['video'].cpu().clone())
        for k, g in enumerate(got, 1):
            assert torch.equal(g, ref[k]), ('pipeline ' + mode, k)
    with pytest.raises(capi.MoogError, match="'huge'"):
        _env(cfg, mod, N, 21, states, dict(cfg['observers'], huge=_renderer(image_size=(4096, 4096), anti_aliasing=4)))
