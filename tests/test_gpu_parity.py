"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the
golden vectors recorded from the unmodified reference.  Needs a B200.

Bars (north_star): overlap / contact pair sets identical (call count, True
count and the order-sensitive hash of the True (slot_a, slot_b) events), state
within 1e-5 relative after a step -- and bit-exact on the scenes whose step
involves only IEEE-exact operations (no sin / cos of a non-zero angle) --
rewards and termination flags identical, frames identical to PILRenderer's.
"""
import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')


def _engine(prog, arrays, n=None):
    from moog_b200.batched_env import Engine
    n = arrays['dyn'].shape[0] if n is None else n
    eng = Engine(prog, n, 'cuda:0')
    eng.state.upload(arrays)
    return eng


def _compare_state(scene, t, prog, dev, ref_arrays, cnt, exact):
    worst = 0.0
    for e in range(cnt.shape[0]):
        live = util.live_mask(prog, cnt[e])
        for k in ('dyn', 'stat'):
            worst = max(worst, util.rel_err(dev[k][e][:, live], ref_arrays[k][e][:, live]))
        vlive = util.live_vertex_mask(prog, cnt[e], ref_arrays['meta'][e])
        worst = max(worst, util.rel_err(dev['vtx'][e][vlive], ref_arrays['vtx'][e][vlive]))
        assert np.array_equal(util.canonical_meta(dev['meta'][e], live),
                              util.canonical_meta(ref_arrays['meta'][e], live)), (scene, t, 'meta')
    if exact:
        assert worst == 0.0, (scene, t, worst)
    else:
        assert worst <= util.RTOL, (scene, t, worst)
    return worst


prog_voff = util.prog_voff


@pytest.mark.parametrize('scene', util.SCENES)
def test_cuda_follows_reference_trajectory(scene):
    """Step by step along the golden trajectory: CUDA vs golden (reference)."""
    g = util.load_golden(scene)
    prog = g['program']
    eng = _engine(prog, util.state_at(g, None, prefix='init'))
    eng.post_reset(rule_noise=util.reset_rule_noise(g))
    dev = eng.state.download()
    util.assert_live_equal(prog, {k: dev[k][0] for k in ('dyn', 'stat', 'vtx', 'cnt', 'meta')},
                           {k: g['reset_' + k] for k in ('dyn', 'stat', 'vtx', 'cnt', 'meta')}, 'reset')
    exact = scene in util.EXACT_SCENES
    T = len(g['reward'])
    for t in range(T):
        noise = g['noise'][t][None] if prog.noise_dim else None
        eng.env_step(g['actions'][t][None], noise=noise, rule_noise=util.rule_noise_at(g, t), auto_reset=False,
                     want_counters=True)
        dev = eng.state.download()
        assert np.array_equal(dev['cnt'][0], g['cnt'][t]), (scene, t)
        ref = {k: g[k][t][None] for k in ('dyn', 'stat', 'vtx', 'meta')}
        _compare_state(scene, t, prog, dev, ref, g['cnt'][t][None], exact)
        assert float(eng.reward[0]) == np.float32(g['reward'][t]), (scene, t)
        assert bool(int(eng.step_type[0]) == 2) == bool(g['last'][t]), (scene, t)
        n_calls, n_true, _, h = eng.counters[0, :4].tolist()
        assert n_calls == g['n_calls'][t], (scene, t, 'overlap call count')
        assert n_true == g['n_true'][t], (scene, t, 'overlap true count')
        assert np.uint64(h & 0xFFFFFFFFFFFFFFFF) == g['true_hash'][t], (scene, t, 'overlap pair set')
        # re-synchronise on the reference state so that one step is compared at a time
        if not exact:
            st = util.state_at(g, t)
            st['envi'] = dev['envi']
            st['envf'] = dev['envf']
            # rule state that lives in the record but not in the reference's sprite objects
            # (Portal._currently_teleporting, portal.py:36-76) stays the device's
            st['meta'][:, 1, :] |= dev['meta'][:, 1, :] & 64
            eng.state.upload(st)


@pytest.mark.parametrize('helper', ['1', '0'])
@pytest.mark.parametrize('scene', util.SCENES)
def test_cuda_matches_oracle_batched(scene, helper, monkeypatch):
    """Every state of the golden trajectory becomes one env of a batch; CUDA and
    the oracle advance the batch 3 steps with the same seeded actions / noise.
    Run with and without the helper warp (second direction of
    _get_collision_vectors computed next to the owner warp)."""
    from oracle.oracle import Oracle
    monkeypatch.setenv('MOOG_HELPER', helper)
    g = util.load_golden(scene)
    prog = g['program']
    T = len(g['reward'])
    parts = [util.state_at(g, t) for t in range(-1, T - 1)]
    arrays = {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}
    n = arrays['dyn'].shape[0]
    rng = np.random.RandomState(7)
    orc = Oracle(prog, arrays)
    eng = _engine(prog, arrays)
    exact = scene in util.EXACT_SCENES
    for step in range(3):
        ad = max(prog.action_dim, 1)
        if any(kind == 'Grid' for _, kind, _, _ in getattr(prog, 'action_layout', [])) or ad == 1:
            actions = rng.randint(0, 5, size=(n, ad)).astype(np.float64)
        else:
            actions = rng.uniform(-1, 1, size=(n, ad))
        noise = rng.uniform(size=(n, prog.K, prog.noise_dim)) if prog.noise_dim else None
        rule_noise = rng.uniform(size=(n, prog.rule_noise_dim)) if prog.rule_noise_dim else None
        if not exact:
            st = orc.arrays()
            st = {k: v.copy() for k, v in st.items()}
            eng.state.upload(st)
        r_ref, st_ref = orc.step(actions, noise=noise, rule_noise=rule_noise)
        eng.env_step(actions, noise=noise, rule_noise=rule_noise, auto_reset=False, want_counters=True)
        dev = eng.state.download()
        assert np.array_equal(dev['cnt'], orc.cnt), (scene, step)
        _compare_state(scene, step, prog, dev, orc.arrays(), orc.cnt, exact)
        assert np.array_equal(eng.reward.cpu().numpy(), r_ref.astype(np.float32)), (scene, step)
        assert np.array_equal(eng.step_type.cpu().numpy(), st_ref), (scene, step)
        c = eng.counters.cpu().numpy()
        assert np.array_equal(c[:, 0], orc.counters[:, 0]), (scene, step, 'overlap call counts')
        assert np.array_equal(c[:, 1], orc.counters[:, 1]), (scene, step, 'overlap true counts')
        assert np.array_equal(c[:, 2], orc.counters[:, 2]), (scene, step, 'resolved collisions')
        assert np.array_equal(c[:, 3], orc.counters[:, 3]), (scene, step, 'overlap pair sets')


@pytest.mark.parametrize('scene', util.SCENES)
def test_cuda_render_matches_reference_frames(scene):
    g = util.load_golden(scene)
    prog = g['program']
    if prog.render is None or len(g['frames']) == 0:
        pytest.skip('scene has no renderer')
    parts = [util.state_at(g, int(t)) for t in g['frame_steps']]
    arrays = {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}
    eng = _engine(prog, arrays)
    out = eng.render().cpu().numpy()
    assert out.shape == g['frames'].shape
    bad = int((out != g['frames']).sum())
    assert bad == 0, (scene, bad)


@pytest.mark.parametrize('scene', util.SCENES)
def test_cuda_overlap_pairs_match_oracle(scene):
    from oracle.oracle import Oracle
    g = util.load_golden(scene)
    prog = g['program']
    T = len(g['reward'])
    parts = [util.state_at(g, t) for t in range(-1, T)]
    arrays = {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}
    orc = Oracle(prog, arrays)
    eng = _engine(prog, arrays)
    names = prog.layer_names
    voff = util.prog_voff(prog)
    big = {n for l, n in enumerate(names) if prog.layer_cap[l] and
           voff[prog.layer_off[l] + 1] - voff[prog.layer_off[l]] > 32}
    for a in names:
        for b in names:
            ref = orc.overlap_pairs(a, b)
            if ref.size == 0:
                continue
            if a in big or b in big:
                # draw-only outlines (MOOG_MAX_OUTLINE): the device refuses to test them
                from moog_b200.capi import MoogError
                with pytest.raises(MoogError):
                    eng.overlap_pairs(a, b)
                continue
            out = eng.overlap_pairs(a, b).cpu().numpy()
            assert np.array_equal(out, ref), (scene, a, b)


@pytest.mark.parametrize('aa', [2, 3])
@pytest.mark.parametrize('scene', util.AA_SCENES)
def test_cuda_render_matches_reference_antialiased_frames(scene, aa):
    g = util.load_golden(scene)
    ga = util.load_golden_aa(scene)
    prog = util.with_anti_aliasing(g, aa)
    parts = [util.state_at(g, int(t)) for t in ga['frame_steps']]
    arrays = {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}
    eng = _engine(prog, arrays)
    out = eng.render().cpu().numpy()
    ref = ga['frames_aa%d' % aa]
    assert out.shape == ref.shape
    bad = int((out != ref).sum())
    assert bad == 0, (scene, aa, bad)


@pytest.mark.parametrize('size', util.BIG_SIZES)
@pytest.mark.parametrize('scene', util.BIG_SCENES)
def test_cuda_render_matches_reference_big_frames(scene, size):
    """Canvases that do not fit one CTA's shared memory are drawn in bands of rows (render_env):
    256 x 256 (the shipped pacman's size), 512 x 512 and a non-square 136 x 200 canvas against
    frames recorded from the reference's PILRenderer; through `moog_render` and through the step
    call's `frames`."""
    g = util.load_golden(scene)
    gb = util.load_golden_big(scene)
    prog = util.with_image_size(g, *size)
    parts = [util.state_at(g, int(t)) for t in gb['frame_steps']]
    arrays = {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}
    eng = _engine(prog, arrays)
    ref = gb['frames_%dx%d' % size]
    out = eng.render().cpu().numpy()
    assert out.shape == ref.shape
    assert int((out != ref).sum()) == 0, (scene, size)
    # the step call's frames of the state it leaves the envs in == a render call afterwards
    eng.frames.zero_()
    eng.env_step(None, auto_reset=False, frames=True)
    got = eng.frames.cpu().numpy().copy()
    again = eng.render(out=torch.zeros_like(eng.frames)).cpu().numpy()
    assert np.array_equal(got, again), (scene, size)


@pytest.mark.gpu
def test_render_env_ranges_and_step_to_host():
    """Frames rendered range by range equal the whole-batch render, and
    `BatchedEnvironment.step_to_host` (chunked render, device-to-host copies on
    a second stream) delivers the same TimeStep as `step` + explicit copies."""
    import torch
    import moog_b200  # noqa: F401
    from moog_b200.batched_env import BatchedEnvironment, TimeStep
    from moog_b200.configs import falling_balls20
    g = util.load_golden('falling_balls20')
    prog = g['program']
    T = len(g['reward'])
    parts = [util.state_at(g, t) for t in range(-1, T - 1)]
    arrays = {k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}
    eng = _engine(prog, arrays)
    whole = eng.render().cpu().numpy().copy()
    eng.frames.zero_()
    n = eng.n
    for first, count in ((0, 7), (7, n - 20), (n - 13, 13)):
        eng.render(first=first, count=count)
    assert np.array_equal(eng.frames.cpu().numpy(), whole)

    cfg = falling_balls20.get_config()
    np.random.seed(4)
    states = [cfg['state_initializer']() for _ in range(8)]
    envs = [BatchedEnvironment(**cfg, num_envs=50, device='cuda:0', seed=9, initial_states=states) for _ in range(2)]
    H = W = 64
    host = TimeStep(torch.empty(50, dtype=torch.int32).pin_memory(), torch.empty(50, dtype=torch.float32).pin_memory(),
                    torch.empty(50, dtype=torch.float32).pin_memory(),
                    {'image': torch.empty((50, H, W, 3), dtype=torch.uint8).pin_memory()})
    act = torch.zeros((50, 1), dtype=torch.float64)
    for step in range(4):
        ts = envs[0].step(act)
        got = envs[1].step_to_host(act, host, chunks=3)
        assert torch.equal(ts.observation['image'].cpu(), got.observation['image']), step
        assert torch.equal(ts.step_type.cpu(), got.step_type), step
        assert torch.equal(torch.nan_to_num(ts.reward.cpu(), nan=-7.), torch.nan_to_num(got.reward, nan=-7.)), step


@pytest.mark.gpu
def test_full_size_batch_matches_oracle_on_a_sample():
    """BASELINE configs[1] at its full size: 4096 falling_balls20 envs stepped 60
    env-steps by the CUDA path (longest-first dispatch, capped residency, helper
    warp, near lists -- everything bench.py exercises, through free fall, the
    first impacts and the piles); a sample of 48 of those envs is stepped by the
    oracle from the same initial states.  Envs are independent, so the sample
    must agree bit for bit, overlap pair sets included."""
    import moog_b200  # noqa: F401
    from moog_b200 import compiler
    from moog_b200.batched_env import Engine
    from moog_b200.configs import falling_balls20
    from oracle.oracle import Oracle
    cfg = falling_balls20.get_config()
    np.random.seed(77)
    states = [cfg['state_initializer']() for _ in range(64)]
    prog = compiler.compile_config(cfg, states)
    pool = compiler.pack_states(prog, states)
    N = 4096
    idx = np.arange(N) % 64
    arrays = {k: np.ascontiguousarray(pool[k][idx]) for k in util.STATE_KEYS}
    # every env gets its own horizontal kick so that the 4096 envs are all different
    arrays['dyn'][:, 2, 4:24] += (np.arange(N)[:, None] % 97) * 1e-5
    eng = Engine(prog, N, 'cuda:0')
    eng.state.upload(arrays)
    eng.post_reset()
    sample = np.arange(7, N, 86)[:48]
    orc = Oracle(prog, {k: arrays[k][sample] for k in util.STATE_KEYS})
    orc.post_reset()
    actions = np.zeros((N, max(prog.action_dim, 1)))
    calls = np.zeros(len(sample), dtype=np.int64)
    for step in range(60):
        eng.env_step(actions, auto_reset=False, want_counters=True)
        orc.step(actions[sample])
        c = eng.counters[torch_index(sample)].cpu().numpy()
        assert np.array_equal(c[:, :4], orc.counters), (step, 'overlap calls / true / resolved / pair-set hash')
        calls += c[:, 2]
        if step % 10 == 9 or step == 59:
            dev = eng.state.download()
            for k in ('dyn', 'vtx', 'cnt'):
                assert np.array_equal(dev[k][sample], getattr(orc, k), equal_nan=(k != 'cnt')), (step, k)
    assert calls.sum() > 1000, 'the sample never reached the contact-heavy phase'
    frames = eng.render().cpu().numpy()
    assert np.array_equal(frames[sample], orc.render())


def torch_index(a):
    import torch
    return torch.as_tensor(a, device='cuda:0')


@pytest.mark.gpu
def test_device_side_reset_sampler():
    """reset_mode='device' (SURVEY section 8 f1): every resetting env draws its generated sprites
    on the device.  The draws respect the factor distributions, the sprites are built like the
    host Sprite builds them (sprite.py:329-424) and the rejection loop of
    sprite_generators.py:69-105 leaves no forbidden overlap."""
    import torch
    import moog_b200  # noqa: F401
    from moog_b200 import compiler as C
    from moog_b200.batched_env import BatchedEnvironment
    from moog_b200.configs import colliding_predators84
    cfg = colliding_predators84.get_config()
    np.random.seed(12)
    states = [cfg['state_initializer']() for _ in range(8)]
    N = 512
    env = BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=5, initial_states=states, reset_mode='device')
    ts = util.device_reset_vs_oracle(env, exact=False)      # (random angles)
    assert bool((ts.step_type == 0).all())
    eng, prog = env.engine, env.program
    st = eng.state.download()
    assert (st['envi'][:, 2] == 0).all(), 'error flags'
    assert (st['cnt'][:, :3] == [4, 5, 1]).all()
    lo = prog.layer_off
    pred = slice(lo[1], lo[1] + 5)
    agent = lo[2]
    # factor ranges (colliding_predators.py:29-52); float32 draws
    x, y = st['dyn'][:, 0, pred], st['dyn'][:, 1, pred]
    scale, aspect = st['stat'][:, 1, pred], st['stat'][:, 2, pred]
    ang, vx, w = st['dyn'][:, 4, pred], st['dyn'][:, 2, pred], st['dyn'][:, 5, pred]
    assert scale.min() >= 0.1 and scale.max() < 0.15 and aspect.min() >= 0.75 and aspect.max() < 1.25
    assert ang.min() >= 0 and ang.max() < 2 * np.pi + 1e-6 and np.abs(vx).max() <= 0.03 and np.abs(w).max() <= 0.05
    for a in (scale, aspect, ang, vx, w):
        assert np.array_equal(a, a.astype(np.float32).astype(np.float64)), 'Continuous factors are float32'
    assert len(np.unique(scale)) > 0.9 * scale.size, 'the envs draw different sprites'
    assert (st['stat'][:, 6:10, pred] == np.array([0., 1., 0.8, 255.])[None, :, None]).all()
    assert (st['meta'][:, 1, pred] & 0x3f == 6).all()           # float32 velocity / angle_vel; the angle is float(angle)
    shapes = st['meta'][:, 0, pred]
    assert set(np.unique(shapes)) == {0, 1, 2, 3, 4}, 'all five shape candidates occur'
    # construction: world vertices, circumscribed radius, inertia as the host Sprite computes them
    hdr = prog.header
    blob = np.frombuffer(prog.blob, dtype=np.uint8)
    n_ops, n_ip, n_ex = int(hdr[C.H_N_OPS]), (int(hdr[C.H_N_IPOOL]) + 1) & ~1, int(hdr[C.H_N_EXPR])
    off = C.HDR_WORDS * 4 + 80 * n_ops
    ipool = np.frombuffer(blob[off:off + 4 * n_ip].tobytes(), dtype='<i4')
    dpool = np.frombuffer(blob[off + 4 * n_ip + 16 * n_ex:].tobytes(), dtype='<f8')
    shape_off = ipool[int(hdr[C.H_SHAPE_TAB]):]
    voff = util.prog_voff(prog)
    worst = 0.0
    for e in range(0, N, 37):
        for s in range(lo[1], lo[1] + 5):
            R = dpool[shape_off[st['meta'][e, 0, s]]:]
            nv = int(R[0])
            assert st['meta'][e, 2, s] == nv
            base = R[6:6 + 2 * nv].reshape(nv, 2)
            px, py = st['dyn'][e, 0, s], st['dyn'][e, 1, s]
            sx = st['stat'][e, 1, s]
            sy = sx * st['stat'][e, 2, s]
            c, sn = np.cos(st['dyn'][e, 4, s]), np.sin(st['dyn'][e, 4, s])
            want = np.stack([c * sx * base[:, 0] + -(sn * sy) * base[:, 1] + px,
                             sn * sx * base[:, 0] + c * sy * base[:, 1] + py], axis=1)
            got = st['vtx'][e, voff[s]:voff[s] + nv]
            worst = max(worst, float(np.abs(got - want).max()))
            rel = want - [px, py]
            assert abs(st['stat'][e, 5, s] - np.sqrt((rel * rel).sum(axis=1)).max()) < 1e-14
            assert abs(st['stat'][e, 3, s] - R[2] * sx * sx) < 1e-18 and abs(st['stat'][e, 4, s] - R[3] * sy * sy) < 1e-18
    assert worst < 1e-15, worst      # cos / sin of the device vs libm: last-bit differences at most
    # rejection: predators are mutually disjoint and clear of the walls, the agent is clear of both
    pp = eng.overlap_pairs('predators', 'predators').cpu().numpy()
    assert not (pp & ~np.eye(5, dtype=bool)[None]).any()
    assert not eng.overlap_pairs('predators', 'walls').cpu().numpy().any()
    assert not eng.overlap_pairs('agent', 'predators').cpu().numpy().any()
    assert not eng.overlap_pairs('agent', 'walls').cpu().numpy().any()
    # episodes end (timeout 200 / contact) and the envs are re-initialised with NEW draws
    first_scale = scale.copy()
    act = torch.zeros((N, 2), dtype=torch.float64)
    for _ in range(205):
        ts = env.step(act)
    st2 = eng.state.download()
    assert (st2['envi'][:, 3] >= 1).all(), 'every env finished at least one episode'
    assert (st2['envi'][:, 2] == 0).all()
    assert (st2['stat'][:, 1, pred] != first_scale).mean() > 0.95
    # same seed -> same draws
    env2 = BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=5, initial_states=states, reset_mode='device')
    env2.reset()
    st3 = env2.engine.state.download()
    for k in ('dyn', 'stat', 'meta', 'cnt'):
        assert np.array_equal(st3[k], st[k]), k
    for e in range(0, N, 61):     # (the vertex slots beyond a sprite's nv keep the template's stale values)
        vlive = util.live_vertex_mask(prog, st['cnt'][e], st['meta'][e])
        assert np.array_equal(st3['vtx'][e][vlive], st['vtx'][e][vlive])


@pytest.mark.gpu
def test_vector_gym_wrapper_and_simulation_snapshot():
    """env_wrappers: the Gym-style protocol over a batch and snapshot / restore
    (reference gym_wrapper.py:48-140, simulation.py:55-83)."""
    import torch
    import moog_b200  # noqa: F401
    from moog_b200.batched_env import BatchedEnvironment
    from moog_b200.configs import colliding_predators84
    from moog_b200.env_wrappers import BatchedSimulation, VectorGymWrapper
    cfg = colliding_predators84.get_config(dict(image_size=(64, 64)))
    np.random.seed(3)
    states = [cfg['state_initializer']() for _ in range(4)]
    env = BatchedEnvironment(**cfg, num_envs=32, device='cuda:0', seed=1, initial_states=states)
    gym = VectorGymWrapper(env)
    assert gym.action_space == [dict(key=None, type='Box', low=-1., high=1., shape=(2,), dtype='float32')]
    assert gym.observation_space['image']['shape'] == (64, 64, 3)
    obs = gym.reset()
    assert obs['image'].shape == (32, 64, 64, 3) and obs['image'].dtype == torch.uint8
    act = torch.full((32, 2), 0.5, dtype=torch.float64)
    obs, reward, done, info = gym.step(act)
    assert reward.shape == (32,) and done.dtype == torch.bool and not bool(done.any())
    assert torch.equal(info['discount'], torch.ones(32, device='cuda:0'))
    sim = BatchedSimulation(env)
    before = env.engine.state.dyn.clone()
    rollout = [sim.sim_step(act).reward.clone() for _ in range(5)]
    assert not torch.equal(env.engine.state.dyn, before) and sim.stack_depth == 5
    sim.sim_pop(0)
    assert torch.equal(env.engine.state.dyn, before) and sim.stack_depth == 0
    again = [sim.sim_step(act).reward.clone() for _ in range(5)]
    assert all(torch.equal(a, b) for a, b in zip(rollout, again)), 'a restored batch replays identically'
    # a real step discards the simulated ones first (simulation.py:64-69)
    first_real = sim.step(act).reward.clone()
    assert sim.stack_depth == 0 and torch.equal(first_real, rollout[0])
    # explicit push / pop
    sim.push()
    mid = env.engine.state.dyn.clone()
    env.step(act)
    sim.pop()
    assert torch.equal(env.engine.state.dyn, mid)


@pytest.mark.gpu
def test_full_size_batch_is_independent_of_the_launch_mode(monkeypatch):
    """All 4096 falling_balls20 envs, 40 env-steps, stepped twice: with the helper warp, the
    32-vertex search tile and the capped residency (the bench's launch), and as a large batch
    would be (one warp per env, 8-vertex tiles, every SM filled).  Dispatch order, residency
    and the split of the directed searches over warps must not change a single bit."""
    import moog_b200  # noqa: F401
    from moog_b200 import compiler
    from moog_b200.batched_env import Engine
    from moog_b200.configs import falling_balls20
    cfg = falling_balls20.get_config()
    np.random.seed(78)
    states = [cfg['state_initializer']() for _ in range(64)]
    prog = compiler.compile_config(cfg, states)
    pool = compiler.pack_states(prog, states)
    N = 4096
    idx = np.arange(N) % 64
    arrays = {k: np.ascontiguousarray(pool[k][idx]) for k in util.STATE_KEYS}
    arrays['dyn'][:, 2, 4:24] += (np.arange(N)[:, None] % 89) * 1e-5
    engines = []
    for helper, cps in ((1, 4), (0, 12)):
        eng = Engine(prog, N, 'cuda:0')
        eng.dev_program.set_option('helper', helper)
        eng.dev_program.set_option('ctas_per_sm', cps)
        eng.state.upload(arrays)
        eng.post_reset()
        engines.append((eng, helper, cps))
    actions = np.zeros((N, max(prog.action_dim, 1)))
    for step in range(40):
        for eng, helper, cps in engines:
            eng.env_step(actions, auto_reset=False, want_counters=True)
        if step % 10 == 9:
            a, b = engines[0][0], engines[1][0]
            for k in ('dyn', 'vtx', 'stat'):
                ta, tb = getattr(a.state, k), getattr(b.state, k)
                same = (ta == tb) | (ta.isnan() & tb.isnan())
                assert bool(same.all()), (step, k)
            assert bool((a.counters[:, :4] == b.counters[:, :4]).all()), (step, 'overlap pair sets')


@pytest.mark.gpu
def test_contact_reward_expression_matches_oracle():
    """ContactReward whose reward_fn reads the two sprites (e.g. first_person_predators_prey.py:133-146,
    `-2. * predator.scale`): traced to an expression, evaluated on the LAST overlapping pair
    (contact_reward.py:86-94) by the CUDA path exactly as by the oracle."""
    import moog_b200  # noqa: F401
    from moog import tasks
    from moog_b200 import compiler
    from moog_b200.configs import colliding_predators84
    from oracle.oracle import Oracle
    cfg = colliding_predators84.get_config(dict(image_size=(64, 64)))
    cfg['task'] = tasks.CompositeTask(
        tasks.ContactReward(reward_fn=lambda s_a, s_p: -2. * s_p.scale + s_a.c0,
                            layers_0='agent', layers_1='predators'), timeout_steps=200)
    np.random.seed(31)
    states = [cfg['state_initializer']() for _ in range(24)]
    prog = compiler.compile_config(cfg, states)
    arr = compiler.pack_states(prog, states)
    arr['stat'][:, 1, prog.layer_off[2]] = 0.3      # a big agent: contacts within a few steps
    orc = Oracle(prog, arr)
    orc.post_reset()
    eng = _engine(prog, arr)
    eng.post_reset()
    rng = np.random.RandomState(3)
    nonzero = 0
    for step in range(40):
        act = rng.uniform(-1, 1, size=(24, 2))
        eng.state.upload({k: v.copy() for k, v in orc.arrays().items()})   # sin / cos scenes: re-sync each step
        r_ref, _ = orc.step(act)
        eng.env_step(act, auto_reset=False)
        got = eng.reward.cpu().numpy()
        assert np.array_equal(got, r_ref.astype(np.float32)), step
        nonzero += int((r_ref != 0).sum())
    assert nonzero > 10


@pytest.mark.gpu
def test_device_reset_sampler_mixture_and_setminus():
    """The factor distributions of first_person_predators_prey.py:37-66 on the device sampler: a
    Mixture of four boundary segments for the position and a SetMinus (square annulus) for the
    velocity."""
    import collections
    import moog_b200  # noqa: F401
    from moog import action_spaces, observers, physics as physics_lib, sprite, tasks
    from moog.state_initialization import distributions as distribs
    from moog.state_initialization import sprite_generators
    from moog_b200.batched_env import BatchedEnvironment
    lo, hi = -0.2, 1.2
    position = distribs.Mixture([
        distribs.Product([distribs.Continuous('y', lo, hi)], x=lo),
        distribs.Product([distribs.Continuous('y', lo, hi)], x=hi),
        distribs.Product([distribs.Continuous('x', lo, hi)], y=lo),
        distribs.Product([distribs.Continuous('x', lo, hi)], y=hi)])
    velocity = distribs.SetMinus(
        distribs.Product([distribs.Continuous('x_vel', -0.03, 0.03), distribs.Continuous('y_vel', -0.03, 0.03)]),
        hold_out=distribs.Product([distribs.Continuous('x_vel', -0.01, 0.01), distribs.Continuous('y_vel', -0.01, 0.01)]))
    factors = distribs.Product([position, velocity, distribs.Continuous('scale', 0.05, 0.1)],
                               shape='square', c0=0.3, c1=1., c2=1.)
    gen = sprite_generators.generate_sprites(factors, num_sprites=6)

    def state_initializer():
        agent = [sprite.Sprite(x=0.5, y=0.5, shape='circle', scale=0.05, c0=0.6, c1=1., c2=1.)]
        return collections.OrderedDict([('agent', agent), ('movers', gen())])

    cfg = dict(state_initializer=state_initializer,
               physics=physics_lib.Physics((physics_lib.Drag(coeff_friction=0.1), 'agent'), updates_per_env_step=2),
               task=tasks.CompositeTask(timeout_steps=20),
               action_space=action_spaces.Joystick(scaling_factor=0.01, action_layers='agent'),
               observers={'image': observers.PILRenderer(image_size=(64, 64), color_to_rgb='hsv_to_rgb')})
    np.random.seed(2)
    states = [state_initializer() for _ in range(2)]
    N = 1024
    env = BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=3, initial_states=states, reset_mode='device')
    util.device_reset_vs_oracle(env, exact=True)      # (no rotated sprite: bit for bit)
    st = env.engine.state.download()
    assert (st['envi'][:, 2] == 0).all() and (st['cnt'][:, :2] == [1, 6]).all()
    s0 = env.program.layer_off[1]
    x, y = st['dyn'][:, 0, s0:s0 + 6].ravel(), st['dyn'][:, 1, s0:s0 + 6].ravel()
    vx, vy = st['dyn'][:, 2, s0:s0 + 6].ravel(), st['dyn'][:, 3, s0:s0 + 6].ravel()
    f32 = lambda a: np.array_equal(a, a.astype(np.float32).astype(np.float64))
    near = lambda a, b: np.abs(a - b) < 1e-12     # (the position is x + the outline's raw centroid, ~1e-17)
    on = np.stack([near(x, lo), near(x, hi), near(y, lo), near(y, hi)], axis=1)
    assert (on.sum(axis=1) == 1).all(), 'every position lies on exactly one boundary segment'
    share = on.mean(axis=0)
    assert np.all(np.abs(share - 0.25) < 0.03), share
    free = np.where(on[:, 0] | on[:, 1], y, x)
    assert free.min() >= lo - 1e-12 and free.max() < hi + 1e-12
    assert np.abs(vx).max() < 0.03 and np.abs(vy).max() < 0.03 and f32(vx) and f32(vy)
    assert not ((np.abs(vx) < 0.01) & (np.abs(vy) < 0.01)).any(), 'the hold-out box is empty'
    assert ((np.abs(vx) < 0.01) | (np.abs(vy) < 0.01)).mean() > 0.3      # ... but only the box, not the cross
    assert (st['meta'][:, 1, s0:s0 + 6] & 0x3f == 2).all()               # float32 velocity array


@pytest.mark.gpu
@pytest.mark.parametrize('helper', ['1', '0'])
@pytest.mark.parametrize('scene', util.SCENES)
def test_step_kernel_draws_the_same_frames_as_the_render_kernel(scene, helper, monkeypatch):
    """`moog_env_step` with `frames`: the step kernel draws the frame of the state it leaves an
    env in from the record in shared memory (owner + helper warp, or the owner alone).  Along
    the golden trajectory the frames must equal what `moog_render` draws from the stored state
    afterwards -- which the tests above pin to PILRenderer's output -- and the state must not
    notice.  A batch of 5 envs draws inside the step kernel wherever one CTA can hold the canvas,
    which every scene here does."""
    g = util.load_golden(scene)
    prog = g['program']
    if prog.render is None:
        pytest.skip('scene has no renderer')
    monkeypatch.setenv('MOOG_HELPER', helper)
    T = min(len(g['reward']), 30)
    n = 5
    arrays = {k: np.concatenate([util.state_at(g, None, prefix='init')[k]] * n, axis=0) for k in util.STATE_KEYS}
    engines = [_engine(prog, arrays), _engine(prog, arrays)]
    assert engines[0].dev_program.step_draws_frames(n), (scene, helper)
    for eng in engines:
        eng.post_reset()
    host = torch.zeros(tuple(engines[0].frames.shape), dtype=torch.uint8).pin_memory()
    for t in range(T):
        noise = np.repeat(g['noise'][t][None], n, axis=0) if prog.noise_dim else None
        rn = util.rule_noise_at(g, t)
        rn = None if rn is None else np.repeat(rn, n, axis=0)
        act = np.repeat(g['actions'][t][None], n, axis=0)
        # engine 0: frames by the step call, alternately into HBM and into pinned host memory
        dst = host if t % 2 else True
        engines[0].env_step(act, noise=noise, rule_noise=rn, auto_reset=False, frames=dst)
        engines[1].env_step(act, noise=noise, rule_noise=rn, auto_reset=False)
        torch.cuda.synchronize()
        got = host.numpy() if t % 2 else engines[0].frames.cpu().numpy()
        ref = engines[1].render().cpu().numpy()
        assert np.array_equal(got, ref), (scene, t, int((got != ref).sum()))
        for k in ('dyn', 'vtx', 'stat'):
            a, b = getattr(engines[0].state, k), getattr(engines[1].state, k)
            assert bool(((a == b) | (a.isnan() & b.isnan())).all()), (scene, t, k)


@pytest.mark.gpu
def test_full_size_batch_frames_from_the_step_call():
    """The bench's launch (4096 falling_balls20 envs: 4 envs per SM, helper warp) with frames:
    the render kernel is launched behind the step kernel with programmatic stream serialization
    and draws the envs in the order they finish, into HBM or straight into pinned host memory;
    the frames equal those of a render call after the step, and `step_to_host` delivers the same
    TimeStep whichever way the frames travel.  Small batches draw inside the step kernel."""
    import moog_b200  # noqa: F401
    from moog_b200.batched_env import BatchedEnvironment, TimeStep
    from moog_b200.configs import falling_balls20
    cfg = falling_balls20.get_config()
    np.random.seed(79)
    states = [cfg['state_initializer']() for _ in range(64)]
    N = 4096
    envs = {m: BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=11, initial_states=states)
            for m in ('mapped', 'device', 'chunked', 'auto')}
    assert not envs['mapped'].engine.dev_program.step_draws_frames(N)
    assert envs['mapped'].engine.dev_program.step_draws_frames(100)
    hosts = {m: TimeStep(torch.empty(N, dtype=torch.int32).pin_memory(), torch.empty(N, dtype=torch.float32).pin_memory(),
                         None, {'image': torch.zeros((N, 64, 64, 3), dtype=torch.uint8).pin_memory()})
             for m in envs}
    act = torch.zeros((N, 1), dtype=torch.float64).pin_memory()
    for step in range(45):
        for m, env in envs.items():
            env.step_to_host(act, hosts[m], frames=m)
        if step % 11 == 0 or step == 44:
            ref = envs['chunked'].engine.render().cpu()
            for m in envs:
                assert torch.equal(hosts[m].observation['image'], ref), (step, m)
                assert torch.equal(hosts[m].step_type, hosts['chunked'].step_type), (step, m)
    # 'auto' timed both transports during its first calls and kept one
    assert envs['auto']._auto_choice in ('mapped', 'chunked')


@pytest.mark.gpu
def test_frames_edge_cases():
    """Edge cases of the frames path: an empty batch, wrong frame buffers, an env whose layers
    are all empty (only the background is drawn), and one env next to 4095 others."""
    import ctypes
    from moog_b200 import capi
    g = util.load_golden('falling_balls20')
    prog = g['program']
    arrays = util.state_at(g, None, prefix='init')
    eng = _engine(prog, arrays)
    eng.post_reset()
    # n_envs = 0: every entry point accepts it and launches nothing
    st = eng.state.struct()
    io = capi.MoogStepIO()
    io.frames = ctypes.c_void_p(eng.frames.data_ptr())
    before = capi.launch_count()
    capi.check(capi.lib().moog_env_step(eng.dev_program.handle, ctypes.byref(st), 0, ctypes.byref(io), None))
    capi.check(capi.lib().moog_render(eng.dev_program.handle, ctypes.byref(st), 0,
                                      ctypes.c_void_p(eng.frames.data_ptr()), None))
    assert capi.launch_count() == before
    # wrong buffers are refused on the host
    with pytest.raises(ValueError):
        eng.env_step(None, frames=torch.zeros((1, 64, 64, 4), dtype=torch.uint8, device='cuda:0'))
    with pytest.raises(ValueError):
        eng.env_step(None, frames=torch.zeros((1, 64, 64, 3), dtype=torch.uint8))      # pageable host memory
    # an env without a single live sprite: background only, through every frame path
    empty = {k: v.copy() for k, v in arrays.items()}
    empty['cnt'][:] = 0
    for n in (1, 4096):
        big = {k: np.repeat(v, n, axis=0) for k, v in (empty if n == 1 else arrays).items()}
        if n > 1:
            big['cnt'][17] = 0
        e2 = _engine(prog, big)
        e2.post_reset()
        e2.env_step(None, auto_reset=False, frames=True)
        torch.cuda.synchronize()
        ref = e2.render(out=torch.zeros_like(e2.frames)).cpu().numpy()
        got = e2.frames.cpu().numpy()
        assert np.array_equal(got, ref), n
        bg = got[0 if n == 1 else 17]
        assert (bg == bg[0, 0]).all(), 'an env without sprites shows the background colour only'


@pytest.mark.gpu
@pytest.mark.parametrize('frames', ['mapped', 'device'])
def test_host_pipeline_delivers_the_same_timesteps(frames):
    """`HostPipeline` (step k+1 enqueued before the host reads step k, TimeSteps in pinned host
    slots) against plain `BatchedEnvironment.step` on a twin environment: every TimeStep of 40
    steps identical, auto-resets included, whichever way the frames travel, at depth 1, 2 and 3."""
    import moog_b200  # noqa: F401
    from moog_b200.batched_env import BatchedEnvironment
    from moog_b200.configs import colliding_predators84
    cfg = colliding_predators84.get_config(dict(image_size=(64, 64)))
    np.random.seed(8)
    states = [cfg['state_initializer']() for _ in range(6)]
    N = 1500
    rng = np.random.RandomState(0)
    acts = [torch.from_numpy(rng.uniform(-1, 1, size=(N, 2))).pin_memory() for _ in range(40)]
    ref_env = BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=21, initial_states=states)
    ref_env.engine.state.envi[:, 0] = 0
    ref = []
    ref_env.reset()
    ref_env.engine.state.envi[:, 0] = torch.arange(N, device='cuda:0', dtype=torch.int32) % 190   # time-outs at every step
    for a in acts:
        ts = ref_env.step(a)
        ref.append((ts.step_type.cpu().clone(), ts.reward.cpu().clone(), ts.discount.cpu().clone(),
                    ts.observation['image'].cpu().clone()))
    assert any(int((r[0] == 0).sum()) > 0 for r in ref[1:]), 'auto-resets happen inside the run'
    for depth in (1, 2, 3):
        env = BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=21, initial_states=states)
        env.reset()
        env.engine.state.envi[:, 0] = torch.arange(N, device='cuda:0', dtype=torch.int32) % 190
        pipe = env.host_pipeline(depth=depth, frames=frames)
        got = []
        scratch = torch.empty_like(acts[0]).pin_memory()
        for k, a in enumerate(acts):
            if k >= depth:
                ts = pipe.collect()
                got.append((ts.step_type.clone(), ts.reward.clone(), ts.discount.clone(), ts.observation['image'].clone()))
            scratch.copy_(a)
            pipe.submit(scratch)
            scratch.fill_(7.0)          # the caller's buffer is free again as soon as submit returns
        while len(got) < len(acts):
            ts = pipe.collect()
            got.append((ts.step_type.clone(), ts.reward.clone(), ts.discount.clone(), ts.observation['image'].clone()))
        for k, (r, g2) in enumerate(zip(ref, got)):
            assert torch.equal(r[0], g2[0]), (depth, k, 'step_type')
            for i in (1, 2):
                assert torch.equal(torch.nan_to_num(r[i], nan=-7.), torch.nan_to_num(g2[i], nan=-7.)), (depth, k, i)
            assert torch.equal(r[3], g2[3]), (depth, k, 'frames')
        with pytest.raises(RuntimeError):
            pipe.collect()


@pytest.mark.gpu
def test_device_reset_sampler_intersection_and_dependent():
    """`Intersection` (distributions.py:211-247: sample one component, reject unless all contain
    the sample) and `DependentDistribution` (:420-470: factors that are a function of the sampled
    ones) on the device sampler."""
    import collections
    import moog_b200  # noqa: F401
    from moog import action_spaces, observers, physics as physics_lib, sprite, tasks
    from moog.state_initialization import distributions as distribs
    from moog.state_initialization import sprite_generators
    from moog_b200.batched_env import BatchedEnvironment
    box = lambda x0, x1, y0, y1: distribs.Product([distribs.Continuous('x', x0, x1), distribs.Continuous('y', y0, y1)])
    position = distribs.Intersection([box(0.1, 0.7, 0.2, 0.9), box(0.4, 0.95, 0.05, 0.6), box(0.0, 1.0, 0.3, 1.0)],
                                     index_for_sampling=0)
    velocity = distribs.DependentDistribution(
        distribs.Continuous('x_vel', -0.03, 0.03),
        dependent_fn=lambda smp: {'y_vel': -0.5 * smp['x_vel'], 'angle_vel': 2. * smp['x_vel'] + 0.01},
        dependent_fn_keys=['y_vel', 'angle_vel'])
    factors = distribs.Product([position, velocity, distribs.Continuous('scale', 0.03, 0.05)], shape='triangle',
                               c0=0.3, c1=1., c2=1.)
    gen = sprite_generators.generate_sprites(factors, num_sprites=5)

    def state_initializer():
        return collections.OrderedDict([('agent', [sprite.Sprite(x=0.5, y=0.02, shape='square', scale=0.02)]),
                                        ('movers', gen())])

    cfg = dict(state_initializer=state_initializer, physics=physics_lib.Physics(updates_per_env_step=1),
               task=tasks.CompositeTask(timeout_steps=10),
               action_space=action_spaces.Joystick(scaling_factor=0.01, action_layers='agent'),
               observers={'image': observers.PILRenderer(image_size=(64, 64), color_to_rgb='hsv_to_rgb')})
    np.random.seed(4)
    states = [state_initializer() for _ in range(2)]
    N = 2048
    env = BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=6, initial_states=states, reset_mode='device')
    util.device_reset_vs_oracle(env, exact=True)      # (no rotated sprite: bit for bit)
    st = env.engine.state.download()
    assert (st['envi'][:, 2] == 0).all() and (st['cnt'][:, :2] == [1, 5]).all()
    s0 = env.program.layer_off[1]
    x, y = st['dyn'][:, 0, s0:s0 + 5].ravel(), st['dyn'][:, 1, s0:s0 + 5].ravel()
    vx, vy, w = (st['dyn'][:, k, s0:s0 + 5].ravel() for k in (2, 3, 5))
    # the intersection of the three boxes is [0.4, 0.7) x [0.3, 0.6); every part of it is reached
    assert x.min() >= 0.4 - 1e-6 and x.max() < 0.7 + 1e-6 and y.min() >= 0.3 - 1e-6 and y.max() < 0.6 + 1e-6
    assert x.min() < 0.42 and x.max() > 0.68 and y.min() < 0.32 and y.max() > 0.58
    # dependent factors: float32 arithmetic on the float32 draw, like NumPy's
    f32 = lambda a: a.astype(np.float32)
    assert np.abs(vx).max() <= 0.03 and len(np.unique(vx)) > 0.9 * vx.size
    assert np.array_equal(f32(vy), f32(-0.5 * vx)) and np.array_equal(vy, f32(vy).astype(np.float64))
    assert np.array_equal(f32(w), f32(2. * vx + 0.01))
    assert (st['meta'][:, 1, s0:s0 + 5] & 0x3f == (2 | (1 << 2))).all()      # float32 velocity and angle_vel


@pytest.mark.gpu
def test_device_reset_sampler_random_sprite_count():
    """`generate_sprites(..., num_sprites=lambda: np.random.randint(2, 5))` (functional_maze.py:146):
    the device sampler draws the count per env and episode."""
    import collections
    import moog_b200  # noqa: F401
    from moog import action_spaces, observers, physics as physics_lib, sprite, tasks
    from moog.state_initialization import distributions as distribs
    from moog.state_initialization import sprite_generators
    from moog_b200.batched_env import BatchedEnvironment
    factors = distribs.Product([distribs.Continuous('x', 0.1, 0.9), distribs.Continuous('y', 0.1, 0.9)],
                               shape='square', scale=0.06, c0=0.5, c1=1., c2=1.)
    gen = sprite_generators.generate_sprites(factors, num_sprites=lambda: np.random.randint(2, 5))

    def state_initializer():
        return collections.OrderedDict([('agent', [sprite.Sprite(x=0.5, y=0.02, shape='square', scale=0.02)]),
                                        ('prey', gen(disjoint=True))])

    cfg = dict(state_initializer=state_initializer, physics=physics_lib.Physics(updates_per_env_step=1),
               task=tasks.CompositeTask(timeout_steps=3),
               action_space=action_spaces.Joystick(scaling_factor=0.01, action_layers='agent'),
               observers={'image': observers.PILRenderer(image_size=(64, 64), color_to_rgb='hsv_to_rgb')})
    np.random.seed(4)
    states = [state_initializer() for _ in range(16)]
    assert {len(s['prey']) for s in states} <= {2, 3, 4}
    N = 3000
    env = BatchedEnvironment(**cfg, num_envs=N, device='cuda:0', seed=6, initial_states=states, reset_mode='device',
                             layer_capacity={'prey': 4})
    util.device_reset_vs_oracle(env, exact=True)      # (no rotated sprite: bit for bit)
    st = env.engine.state.download()
    counts = st['cnt'][:, 1]
    share = np.array([(counts == c).mean() for c in (2, 3, 4)])
    assert share.sum() == 1.0 and np.all(np.abs(share - 1 / 3) < 0.04), share
    # the sprites that exist are disjoint
    pp = env.engine.overlap_pairs('prey', 'prey').cpu().numpy()
    for e in range(0, N, 17):
        c = counts[e]
        assert not (pp[e, :c, :c] & ~np.eye(c, dtype=bool)).any()
    first = counts.copy()
    import torch
    for _ in range(5):
        env.step(torch.zeros((N, 2), dtype=torch.float64))
    again = env.engine.state.download()['cnt'][:, 1]
    assert (again != first).mean() > 0.5, 'a new count is drawn every episode'


@pytest.mark.gpu
@pytest.mark.parametrize('scene,n_envs', [('colliding_predators84', 16384), ('cleanup64', 8192), ('pacman64', 8192),
                                          ('synthetic32', 131072)])
def test_full_size_other_baseline_configs_match_oracle_on_a_sample(scene, n_envs):
    """BASELINE configs[2..4] and the synthetic stress scene AT THEIR FULL SIZES (16 384 / 8 192 / 8 192 /
    131 072 envs on one GPU -- the launch modes, residencies and record sizes `bench.py --scene` exercises): the
    batch is stepped by the CUDA path with seeded per-env actions / noise; 40 of its envs are stepped by the
    oracle from the same initial states.  Envs are independent (the size-independent property), so the sample
    must agree: counts, dtype flags and overlap call statistics exactly, attributes and outlines within 1e-5
    (bit for bit where no sprite rotates), frames identical at the end."""
    import importlib
    import moog_b200  # noqa: F401
    from moog_b200 import compiler
    from moog_b200.batched_env import Engine
    from oracle.oracle import Oracle
    cfg = importlib.import_module('moog_b200.configs.' + scene).get_config()
    np.random.seed(31)
    states = [cfg['state_initializer']() for _ in range(24)]
    prog = compiler.compile_config(cfg, states)
    pool = compiler.pack_states(prog, states)
    N = n_envs
    rng = np.random.RandomState(5)
    idx = rng.randint(0, 24, size=N)
    arrays = {k: np.ascontiguousarray(pool[k][idx]) for k in util.STATE_KEYS}
    eng = Engine(prog, N, 'cuda:0')
    eng.state.upload(arrays)
    eng.post_reset()
    sample = np.sort(rng.choice(N, size=40, replace=False))
    orc = Oracle(prog, {k: arrays[k][sample] for k in util.STATE_KEYS})
    orc.post_reset()
    ad = max(prog.action_dim, 1)
    grid = any(kind == 'Grid' for _, kind, _, _ in prog.action_layout)
    worst = 0.0
    for step in range(6):
        act = rng.randint(0, 5, size=(N, ad)).astype(np.float64) if grid else rng.uniform(-1, 1, size=(N, ad))
        noise = rng.uniform(size=(N, prog.K * prog.noise_dim)) if prog.noise_dim else None
        rn = rng.uniform(size=(N, prog.rule_noise_dim)) if prog.rule_noise_dim else None
        eng.env_step(act, noise=noise, rule_noise=rn, auto_reset=False, want_counters=True)
        r_ref, st_ref = orc.step(act[sample],
                                 noise=None if noise is None else noise[sample].reshape(len(sample), prog.K, prog.noise_dim),
                                 rule_noise=None if rn is None else rn[sample])
        assert np.array_equal(eng.step_type[torch_index(sample)].cpu().numpy(), st_ref), (scene, step)
        c = eng.counters[torch_index(sample)].cpu().numpy()
        assert np.array_equal(c[:, :2], orc.counters[:, :2]), (scene, step, 'overlap calls / true')
        got = {k: getattr(eng.state, k)[torch_index(sample)].cpu().numpy() for k in ('dyn', 'stat', 'meta', 'vtx', 'cnt')}
        assert np.array_equal(got['cnt'], orc.cnt), (scene, step)
        for e in range(len(sample)):
            live = util.live_mask(prog, orc.cnt[e])
            assert np.array_equal(util.canonical_meta(got['meta'][e], live), util.canonical_meta(orc.meta[e], live)), (scene, step, e)
            vlive = util.live_vertex_mask(prog, orc.cnt[e], orc.meta[e])
            worst = max(worst, util.rel_err(got['dyn'][e][:, live], orc.dyn[e][:, live]),
                        util.rel_err(got['stat'][e][:, live], orc.stat[e][:, live]),
                        util.rel_err(got['vtx'][e][vlive], orc.vtx[e][vlive]))
        assert worst <= util.RTOL, (scene, step, worst)
    st = eng.state.download() if N <= 16384 else None
    if st is not None:
        assert (st['envi'][:, 2] == 0).all()
    if prog.render is not None and worst == 0.0:
        frames = eng.render()[torch_index(sample)].cpu().numpy()
        assert np.array_equal(frames, orc.render())

