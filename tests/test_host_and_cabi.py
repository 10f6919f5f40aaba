"""CPU-side tests: the C-ABI library loads and exports what include/moog_b200.h
declares, the host geometry agrees with the oracle, the product path refuses to
run without a GPU, the env-sharding logic works over 2 gloo ranks."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from tests import util

ROOT = util.ROOT


def _header_functions():
    text = open(os.path.join(ROOT, 'include', 'moog_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(moog_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    import moog_b200  # noqa: F401
    from moog_b200 import build, capi
    lib = build.build()
    L = ctypes.CDLL(lib)
    declared = _header_functions()
    assert len(declared) >= 10
    for name in declared:
        assert hasattr(L, name), name
    assert sorted(capi.SYMBOLS) == declared


def test_program_blob_is_validated_without_a_gpu():
    """moog_program_create rejects malformed blobs before touching CUDA."""
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    L = capi.lib()
    h = ctypes.c_void_p()
    junk = ctypes.create_string_buffer(b'\0' * 512, 512)
    assert L.moog_program_create(junk, 512, ctypes.byref(h)) == -1
    assert L.moog_strerror(-1).decode().startswith('invalid')


def test_host_geometry_matches_oracle():
    """moog_host_paths_overlap (host Sprite.overlaps_sprite) vs the oracle's
    restatement of Path.intersects_path on random near-touching polygons."""
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    from oracle.oracle import lib as orc_lib
    L, O = capi.lib(), orc_lib()
    O.orc_path_intersects_filled.restype = ctypes.c_int
    rng = np.random.RandomState(0)
    n_true = 0
    for trial in range(4000):
        polys = []
        for _ in range(2):
            n = rng.randint(3, 12)
            ang = np.sort(rng.uniform(0, 2 * np.pi, n))
            r = rng.uniform(0.05, 0.2)
            c = rng.uniform(0.3, 0.7, 2)
            p = c + r * np.stack([np.cos(ang), np.sin(ang)], 1)
            polys.append(np.ascontiguousarray(np.vstack([p, p[:1]])))
        a, b = polys
        ra = L.moog_host_paths_overlap(a.ctypes.data_as(ctypes.c_void_p), len(a),
                                       b.ctypes.data_as(ctypes.c_void_p), len(b))
        rb = O.orc_path_intersects_filled(a.ctypes.data_as(ctypes.c_void_p), len(a),
                                          b.ctypes.data_as(ctypes.c_void_p), len(b))
        assert bool(ra) == bool(rb), trial
        n_true += bool(ra)
    assert 200 < n_true < 3800


def test_device_path_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    from moog_b200.batched_env import Engine
    g = util.load_golden('pong')
    with pytest.raises(capi.MoogError):
        Engine(g['program'], 4, 'cuda:0')


@pytest.mark.gpu
def test_set_option_takes_the_launch_options_and_refuses_other_names():
    """moog_program_set_option changes "helper", "ctas_per_sm", "trace_times" and "seed" of a live
    program and returns MOOG_E_INVAL for any other name, such as the launch options that used to
    select a code path or a size the library picks itself."""
    import moog_b200  # noqa: F401
    from moog_b200 import capi
    prog = capi.DeviceProgram(util.load_golden('falling_balls20')['program'].blob)
    L = capi.lib()

    def set_option(name, value):
        return L.moog_program_set_option(prog.handle, name.encode(), value)

    for name, value in (('helper', 0), ('ctas_per_sm', 3), ('trace_times', 1), ('seed', 7)):
        assert set_option(name, value) == 0, name
    assert prog.step_launch_info(4096)[:2] == (3, 1)
    for name, value in (('helper', -1), ('ctas_per_sm', 0), ('trace_times', 0), ('seed', 0)):
        assert set_option(name, value) == 0, name
    for name in ('tail_render', 'fused_render', 'smem_pad', 'render_epb', 'tail_ctas_per_sm', 'tail_busy_thr'):
        assert set_option(name, 1) == capi.E_INVAL, name
    prog.close()


def test_product_package_never_touches_the_oracle():
    pkg = os.path.join(ROOT, 'moog.github.io_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.cpp', '.h')):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', text, flags=re.M), f
                assert 'libmoog_oracle' not in text, f


def test_compile_shipped_style_config_and_pack_states():
    import moog_b200  # noqa: F401
    from moog_b200 import compiler
    from moog_b200.configs import falling_balls20
    np.random.seed(3)
    cfg = falling_balls20.get_config()
    states = [cfg['state_initializer']() for _ in range(3)]
    prog = compiler.compile_config(cfg, states)
    assert prog.layer_names == ['walls', 'balls', 'agent']
    assert prog.n_slots == 24 and prog.K == 20 and prog.n_vtx == 4 * 4 + 20 * 30
    arr = compiler.pack_states(prog, states)
    assert arr['dyn'].shape == (3, 6, 24) and arr['vtx'].shape == (3, 616, 2)
    assert (arr['cnt'][:, :3] == [4, 20, 0]).all()
    hdr = np.frombuffer(prog.blob[:256], dtype='<i4')
    assert hdr[compiler.H_MAGIC] == compiler.MAGIC and hdr[compiler.H_BYTES] == len(prog.blob)


_WORKER = r'''
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
import moog_b200
from moog_b200 import dist as mdist
from oracle.oracle import Oracle
from tests import util
rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:{port}', rank=rank, world_size=world)
g = util.load_golden('falling_balls20')
prog = g['program']
T = 10
parts = [util.state_at(g, t) for t in range(T)]
arrays = {{k: np.concatenate([p[k] for p in parts], axis=0) for k in util.STATE_KEYS}}
lo, hi = mdist.shard_range(T, rank, world)
mine = {{k: v[lo:hi] for k, v in arrays.items()}}
orc = Oracle(prog, mine)
stats = torch.zeros(4, dtype=torch.float64)
for step in range(3):
    r, st = orc.step(np.zeros((hi - lo, 1)))
    stats[0] += float(r.sum()); stats[3] += hi - lo
    stats[2] += float((st == 2).sum())
mdist.reduce_stats(stats)
slowest = mdist.max_over_ranks(1.0 + rank)
chk = torch.tensor([float(orc.dyn.sum())], dtype=torch.float64)
dist.all_reduce(chk)
if rank == 0:
    full = Oracle(prog, arrays)
    for step in range(3):
        full.step(np.zeros((T, 1)))
    assert stats[3] == 3 * T, stats
    assert slowest == float(world), slowest
    assert abs(chk.item() - full.dyn.sum()) < 1e-9, (chk.item(), full.dyn.sum())
    print('OK')
dist.destroy_process_group()
'''


def test_env_sharding_over_two_gloo_ranks(tmp_path):
    """world_size-2 run of the N>1 host logic on CPU: contiguous env shards, the
    stats all_reduce, max-over-ranks timing; sharded result == unsharded."""
    import socket
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / 'worker.py'
    script.write_text(_WORKER.format(root=ROOT, port=port))
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE='2', MASTER_ADDR='127.0.0.1',
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=240) for p in procs]
    for p, (o, e) in zip(procs, outs):
        assert p.returncode == 0, e[-2000:]
    assert 'OK' in outs[0][0]


def test_shard_range_partitions():
    import moog_b200  # noqa: F401
    from moog_b200 import dist as mdist
    for n in (0, 1, 7, 4096, 1 << 20):
        for w in (1, 2, 3, 8):
            spans = [mdist.shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            for a, b in zip(spans[:-1], spans[1:]):
                assert a[1] == b[0]
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_maze_record_round_trips_through_wall_sprites():
    """Maze -> wall sprites -> host_maze.maze_matrix (Maze.from_state restated,
    maze.py:38-84) gives the maze back; the record packs rows as bit masks."""
    import moog_b200  # noqa: F401
    from moog import maze_lib
    from moog_b200 import host_maze
    np.random.seed(11)
    for size, ambient in ((8, 12), (10, 12), (6, 7)):
        m = maze_lib.generate_random_maze_matrix(size=size, ambient_size=ambient)
        # generator contract (maze_generators.py:96-110): no open 2x2 block, no dead end
        opened = 1 - m
        assert not (opened[:-1, :-1] * opened[1:, :-1] * opened[:-1, 1:] * opened[1:, 1:]).any()
        pad = np.pad(opened, 1)
        nb = pad[:-2, 1:-1] + pad[2:, 1:-1] + pad[1:-1, :-2] + pad[1:-1, 2:]
        assert (nb[opened == 1] >= 2).all()
        maze = maze_lib.Maze(np.flip(m, axis=0))
        walls = maze.to_sprites(c0=0., c1=0., c2=0.8)
        got = host_maze.maze_matrix(walls)
        assert np.array_equal(got, maze.maze.astype(int)), (size, ambient)
        rec = host_maze.maze_record(walls)
        assert rec[0] == ambient
        for j in range(ambient):
            assert int(rec[1 + j]) == sum(int(maze.maze[j, i]) << i for i in range(ambient))


def test_pacman64_compiles_and_steps_on_the_oracle():
    """BASELINE config 4 through this repo's own MOOG-compatible host package:
    RandomMazeWalk / MazePhysics / Grid / VanishOnContact / the `unglue`
    ConditionalRule lower to device ops, and the CPU oracle steps the packed
    states without leaving the maze grid (maze_physics.py:93-104)."""
    import moog_b200  # noqa: F401
    from moog_b200 import compiler
    from moog_b200.configs import pacman64
    from oracle.oracle import Oracle
    np.random.seed(5)
    cfg = pacman64.get_config(0)
    states = [cfg['state_initializer']() for _ in range(3)]
    prog = compiler.compile_config(cfg, states)
    assert prog.layer_names == ['walls', 'prey', 'ghosts', 'agent'] and prog.K == 1
    assert prog.noise_dim == 4 * 2 and 'walls' in prog.maze_offsets
    kinds = [o['kind'] for o in prog.ops]
    assert compiler.F_MAZE_WALK in kinds and compiler.C_MAZE_PHYSICS in kinds and compiler.SC_FIRST in kinds
    arr = compiler.pack_states(prog, states)
    orc = Oracle(prog, arr)
    orc.post_reset()
    rng = np.random.RandomState(0)
    prey0 = orc.cnt[:, 1].copy()
    moved = np.zeros(3, dtype=bool)
    for _ in range(80):
        p0 = orc.dyn[:, 0:2, prog.layer_off[3]].copy()
        orc.step(rng.randint(0, 4, size=(3, 1)).astype(np.float64), noise=rng.uniform(size=(3, 1, prog.noise_dim)))
        moved |= (orc.dyn[:, 0:2, prog.layer_off[3]] != p0).any(axis=1)
    assert (orc.envi[:, 2] == 0).all()          # no MOOG_ERR_* flag
    assert moved.all() and (orc.cnt[:, 1] < prey0).all()   # the agents move and eat prey
    # the agent stays on the maze grid: one coordinate on a grid line
    grid = 1. / 12
    pos = orc.dyn[:, 0:2, prog.layer_off[3]]
    off = np.abs((pos / grid - 0.5) - np.round(pos / grid - 0.5))
    assert (off.min(axis=1) < 1e-3).all()


def test_host_maze_matches_reference_from_state():
    """host_maze on the wall sprites of the reference's pacman initial state recorded in tests/golden
    (rebuilt as host sprites from their outlines and factors) gives the maze record stored with that
    trajectory -- the record under which the oracle and the GPU reproduce the reference's MazePhysics /
    RandomMazeWalk steps (test_oracle_vs_golden, test_gpu_parity)."""
    import moog_b200  # noqa: F401
    from moog import sprite as sprite_lib
    from moog_b200 import host_maze
    from tests import util
    g = util.load_golden('pacman')
    prog = g['program']
    walls = prog.layer_index('walls')
    for prefix in ('init', 'reset'):
        dyn, stat, meta, cnt = (g[prefix + '_' + k] for k in ('dyn', 'stat', 'meta', 'cnt'))
        sprites = []
        for s in range(prog.layer_off[walls], prog.layer_off[walls] + int(cnt[walls])):
            k = meta[0, s]
            sprites.append(sprite_lib.Sprite(x=dyn[0, s], y=dyn[1, s], shape=g['shape_verts'][k, :g['shape_nv'][k]],
                                             angle=dyn[4, s], scale=stat[1, s], aspect_ratio=stat[2, s]))
        rec = host_maze.maze_record(sprites)
        envf = g[prefix + '_envf']
        n = int(rec[0])
        assert n > 1 and host_maze.maze_matrix(sprites).shape == (n, n)
        found = [o for o in range(len(envf) - n) if np.array_equal(envf[o:o + 1 + n], rec[:1 + n])]
        assert found, (prefix, rec[:1 + n], envf)


@pytest.mark.reference
def test_host_maze_matches_reference_checkout():
    """With a checkout of the original project: host_maze.maze_matrix == the reference's
    Maze.from_state on the reference's own pacman initial states (levels 0 and 1)."""
    import subprocess
    import sys
    code = r'''
import sys
sys.path.insert(0, %r)
from oracle import refenv
refenv.activate()
import numpy as np, importlib
import moog_b200
from moog_b200 import host_maze
from moog import maze_lib
np.random.seed(21)
for level in (0, 1):
    cfg = importlib.import_module('moog_demos.example_configs.pacman').get_config(level)
    for _ in range(3):
        st = cfg['state_initializer']()
        ref = maze_lib.Maze.from_state(st, maze_layer='walls').maze
        assert np.array_equal(host_maze.maze_matrix(st['walls']), ref)
print('OK')
''' % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))),)
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and 'OK' in out.stdout, out.stdout[-1000:] + out.stderr[-2000:]


@pytest.mark.parametrize('name,slots,K,action_dim', [
    ('colliding_predators84', 10, 10, 2), ('cleanup64', 31, 5, 6), ('synthetic32', 32, 10, 1)])
def test_baseline_configs_of_this_package_compile_and_step(name, slots, K, action_dim):
    """The BASELINE.json configs shipped in moog_b200/configs (this repo's own
    MOOG-compatible host package, no reference needed) compile and step on the oracle."""
    import importlib
    import moog_b200  # noqa: F401
    from moog_b200 import compiler
    from oracle.oracle import Oracle
    cfg = importlib.import_module('moog_b200.configs.' + name).get_config()
    np.random.seed(2)
    states = [cfg['state_initializer']() for _ in range(3)]
    prog = compiler.compile_config(cfg, states)
    assert (prog.n_slots, prog.K, max(prog.action_dim, 1)) == (slots, K, action_dim)
    arr = compiler.pack_states(prog, states)
    orc = Oracle(prog, arr)
    orc.post_reset()
    rng = np.random.RandomState(1)
    before = orc.dyn.copy()
    for _ in range(5):
        orc.step(rng.uniform(-1, 1, size=(3, action_dim)),
                 rule_noise=rng.uniform(size=(3, max(prog.rule_noise_dim, 1))) if prog.rule_noise_dim else None)
    assert (orc.envi[:, 2] == 0).all() and not np.array_equal(orc.dyn, before)
    if prog.render is not None:
        assert orc.render().shape == (3, prog.render['height'], prog.render['width'], 3)


def test_reset_sampler_lowering():
    """compile_config(reset_sampler=True) traces the state initializer (this repo's
    sprite_generators record their calls) and lowers every generate_sprites group to a
    MOOG_Z_GENERATE op; what cannot run on the device is refused at compile time."""
    import moog_b200  # noqa: F401
    from moog_b200 import compiler as C
    from moog_b200.configs import colliding_predators84, pacman64
    np.random.seed(8)
    cfg = colliding_predators84.get_config()
    states = [cfg['state_initializer']() for _ in range(6)]
    prog = C.compile_config(cfg, states, reset_sampler=True)
    start, count = prog.sections['reset']
    ops = prog.ops[start:start + count]
    assert [o['kind'] for o in ops] == [C.Z_GENERATE, C.Z_GENERATE]
    pred, agent = ops
    assert pred['i'][0] == prog.layer_off[1] and pred['i'][1] == 5 and pred['i'][3] == 4 and pred['flags'] & C.FL_DISJOINT
    assert agent['i'][0] == prog.layer_off[2] and agent['i'][1] == 1 and agent['i'][3] == 9 and not agent['flags'] & C.FL_DISJOINT
    # float32 velocity and angle_vel; the angle is float(angle) (sprite.py:310), never float32 at birth
    assert pred['i'][5] == C.SF_VEL32 | (1 << C.SF_ANGVEL_SHIFT) and agent['i'][5] == 0
    assert len(prog.reset_shapes) == 6          # 5 predator candidates + the agent's circle
    tab = prog.ipool[pred['i'][4]:pred['i'][4] + 3 * C.Z_N_ATTRS]
    kinds = tab[0::3]
    assert kinds[0] == C.ZK_UNIFORM32 and kinds[C.Z_SHAPE_ATTR] == C.ZK_DISCRETE and kinds[6] == C.ZK_CONST
    lo_hi = prog.dpool[tab[3 * 7 + 1]:tab[3 * 7 + 1] + 2]       # scale ~ U[0.1, 0.15)
    assert lo_hi == [0.1, 0.15]
    hdr = np.frombuffer(prog.blob[:256], dtype='<i4')
    assert hdr[C.H_N_RESET] == 2 and hdr[C.H_N_DPOOL] == len(prog.dpool) and hdr[C.H_BYTES] == len(prog.blob)
    # a program compiled without the sampler carries no reset section (old blobs stay valid)
    plain = C.compile_config(cfg, states)
    assert np.frombuffer(plain.blob[:256], dtype='<i4')[C.H_N_RESET] == 0
    # an initializer that never calls generate_sprites (pacman builds its sprites by hand) is refused
    pcfg = pacman64.get_config(0)
    pstates = [pcfg['state_initializer']() for _ in range(2)]
    with pytest.raises(C.CompileError):
        C.compile_config(pcfg, pstates, reset_sampler=True)


def test_reward_function_lowering():
    """constant rewards stay constants; functions of the two sprites become expressions;
    Python branches on sprite values become selects, numeric metadata becomes columns."""
    import moog_b200  # noqa: F401
    from moog_b200 import lambdas
    assert lambdas.pair_reward(-5) == (-5.0, None)
    assert lambdas.pair_reward(lambda a, b: 1.5) == (1.5, None)
    const, code = lambdas.pair_reward(lambda a, b: -2. * b.scale)
    assert const == 0.0 and [c[0] for c in code] == [lambdas.X_CONST, lambdas.X_ATTR1, lambdas.X_MUL]
    # a Python branch on a sprite value: both sides are traced and folded into a select
    const, code = lambdas.pair_reward(lambda a, b: 1. if b.c0 < 128 else -1.)
    assert const == 0.0 and [c[0] for c in code] == [lambdas.X_ATTR1, lambdas.X_CONST, lambdas.X_LT, lambdas.X_CONST,
                                                      lambdas.X_CONST, lambdas.X_SELECT]
    # metadata is only readable while a program is being compiled (its keys become columns of the record)
    with pytest.raises(lambdas.LoweringError):
        lambdas.pair_reward(lambda a, b: a.metadata['true_contact_color'])
    keys = []
    with lambdas.metadata_columns(keys):
        const, code = lambdas.pair_reward(lambda a, b: a.metadata['true_contact_color'])
    assert keys == ['true_contact_color'] and code == [(lambdas.X_ATTR0, lambdas.AT_META0, 0.0)]


_VANISH_RANGE = [-1.2, 2.2]


def _should_vanish(s):
    """first_person_predators_prey.py:196-199 verbatim in structure: vector comparisons,
    products of masks, builtin any(), Python `or`."""
    pos_too_small = (s.position < _VANISH_RANGE[0]) * (s.velocity < 0.)
    pos_too_large = (s.position > _VANISH_RANGE[1]) * (s.velocity > 0.)
    return any(pos_too_small) or any(pos_too_large)


def _wrap_position(s):
    s.position = np.remainder(s.position, 1)


def test_vector_valued_and_boolean_lambdas_lower_to_expressions():
    """Sprite callables that use position / velocity as vectors, NumPy ufuncs on them, the
    builtins any / all and Python's and / or / not are traced (after an AST rewrite of the
    boolean constructs) to the postfix VM; evaluated here with a tiny interpreter."""
    import moog_b200  # noqa: F401
    from moog_b200 import lambdas as L

    def run(code, attrs):
        st = []
        for op, arg, c in code:
            if op == L.X_CONST:
                st.append(c)
            elif op == L.X_ATTR0:
                st.append(attrs[L.ATTRS[arg]])
            elif op == L.X_NOT:
                st.append(float(not st.pop()))
            elif op == L.X_STORE:
                attrs[L.ATTRS[arg]] = st.pop()
            elif op == L.X_STORE_POS:
                attrs['y'] = st.pop()
                attrs['x'] = st.pop()
            else:
                b, a = st.pop(), st.pop()
                st.append(float({L.X_LT: a < b, L.X_LE: a <= b, L.X_GT: a > b, L.X_GE: a >= b, L.X_EQ: a == b,
                                 L.X_NE: a != b, L.X_AND: bool(a) and bool(b), L.X_OR: bool(a) or bool(b),
                                 L.X_ADD: a + b, L.X_SUB: a - b, L.X_MUL: a * b, L.X_DIV: a / b if b else 0.,
                                 L.X_MOD: a % b if b else 0.}[op]))
        return st[-1] if st else None

    code = L.compile_sprite_predicate(_should_vanish)
    base = dict(x=0.5, y=0.5, x_vel=0.01, y_vel=-0.01)
    assert run(code, dict(base)) == 0.0
    assert run(code, dict(base, y=-1.3)) == 1.0           # below the range and moving down
    assert run(code, dict(base, y=-1.3, y_vel=0.01)) == 0.0
    assert run(code, dict(base, x=2.3)) == 1.0            # right of the range and moving right
    attrs = dict(x=1.25, y=-0.25)
    run(L.compile_modifier(_wrap_position), attrs)
    assert attrs == dict(x=0.25, y=0.75)
    code = L.compile_sprite_predicate(lambda s: s.c2 > 0.6 and not s.mass == 1)
    assert run(code, dict(c2=0.7, mass=2.)) == 1.0 and run(code, dict(c2=0.7, mass=1.)) == 0.0
    # a Python branch on a sprite value: every path is traced, the results folded into a select
    code = L.compile_sprite_predicate(lambda s: 1. if s.c0 < 128 else -1.)
    assert L.X_SELECT in [op for op, _, _ in code]
    # ... but not in a callable with effects
    def _branching_modifier(s):
        if s.c0 < 128:
            s.c0 = 255
    with pytest.raises(L.LoweringError):
        L.compile_modifier(_branching_modifier)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU port on the host cores, the one place besides the tests
    where bench.py executes oracle/) prints exactly one JSON line with the keys the driver reads;
    under torchrun every rank but 0 exits without work."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0']
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'env-steps/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['steps'] == 1 and d['n_gpus'] == 1
    assert d['config']['workload'] == 'falling_balls20'
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['cpu_baseline']['value'] == d['value'] == d['e2e']['value']
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    other = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root, env=env)
    assert other.returncode == 0 and other.stdout.strip() == ''


def test_step_to_host_auto_policy_keeps_the_faster_transport():
    """Host logic of `step_to_host(frames='auto')` (no GPU needed): the first calls alternate
    between the mapped host image and chunked copies, the first call of each is a warm-up, and
    the transport with the smaller best time is kept; pageable host images always use 'device'."""
    import moog_b200  # noqa: F401
    from moog_b200.batched_env import BatchedEnvironment

    class Img(object):
        def __init__(self, pinned):
            self._p = pinned

        def is_pinned(self):
            return self._p

    def fresh():
        env = object.__new__(BatchedEnvironment)
        env._auto_choice, env._auto_calls = None, 0
        env._auto_times = {'mapped': [], 'chunked': []}
        return env

    for cost, winner in (({'mapped': 5.0, 'chunked': 5.5}, 'mapped'), ({'mapped': 16.6, 'chunked': 11.0}, 'chunked')):
        env = fresh()
        seen = []
        for call in range(12):
            mode = env._auto_frames(Img(True))
            seen.append(mode)
            # the very first call of each transport is slow (allocations, first launches)
            env._auto_record(mode, cost[mode] * (10.0 if call < 2 else 1.0))
        assert seen[:8] == ['mapped', 'chunked'] * 4
        assert env._auto_choice == winner and seen[8:] == [winner] * 4
    assert fresh()._auto_frames(Img(False)) == 'device'
    assert fresh()._auto_frames(None) == 'device'


def test_impure_config_callables_are_refused():
    """A modifier / reward / interval that draws random numbers would be traced ONCE and frozen into
    a constant for every env and step (round-1 advisor finding; e.g. match_to_sample.py:227-228).
    The compiler refuses it; deterministic callables still lower."""
    import moog_b200  # noqa: F401
    from moog import game_rules
    from moog_b200 import compiler, lambdas
    from moog_b200.configs import timed_center

    def _kick(s):
        s.velocity = np.random.uniform(-0.25, 0.25, size=(2,))

    with pytest.raises(lambdas.LoweringError, match='random'):
        lambdas.compile_modifier(_kick)
    with pytest.raises(lambdas.LoweringError, match='random'):
        lambdas.pair_reward(lambda a, b: np.random.rand())
    state = np.random.get_state()
    lambdas.compile_modifier(lambda s: setattr(s, 'opacity', 128))
    assert np.random.get_state()[1].tolist() == state[1].tolist(), 'tracing consumes no random numbers'
    assert np.random.uniform.__name__ == 'uniform', 'numpy.random is restored after tracing'

    cfg = timed_center.get_config()
    np.random.seed(1)
    states = [cfg['state_initializer']()]
    compiler.compile_config(cfg, states)                       # fixed intervals: fine
    rules = list(cfg['game_rules'])
    rules[1] = game_rules.TimedRule(lambda: (5, 6) if np.random.rand() < 0.5 else (7, 8), game_rules.VanishByFilter('cue'))
    cfg['game_rules'] = tuple(rules)
    with pytest.raises(compiler.CompileError, match='random step interval'):
        compiler.compile_config(cfg, states)
    # rules nested deeper than the device's block stack are refused instead of silently skipped
    inner = game_rules.VanishByFilter('cue')
    for _ in range(5):
        inner = game_rules.ConditionalRule(lambda state: True, inner)
    cfg['game_rules'] = (inner,)
    with pytest.raises(compiler.CompileError, match='nested deeper'):
        compiler.compile_config(cfg, states)


def test_program_blobs_are_validated():
    """moog_program_validate (what moog_program_create runs first; no GPU needed): every golden program
    and every config of this package passes; blobs with a section, pool index, layer id, expression
    start, op kind or outline offset out of range are MOOG_E_INVAL, not an out-of-bounds read."""
    import ctypes
    import glob
    import importlib
    import moog_b200  # noqa: F401
    from moog_b200 import capi, compiler as C
    L = capi.lib()

    def check(blob):
        buf = (ctypes.c_uint8 * len(blob)).from_buffer_copy(bytes(blob))
        return L.moog_program_validate(ctypes.cast(buf, ctypes.c_void_p), len(blob))

    blobs = []
    for path in sorted(glob.glob(os.path.join(util.GOLDEN, '*.npz'))):
        g = np.load(path)
        if 'blob' in g:
            blobs.append((os.path.basename(path), bytes(bytearray(g['blob']))))
    for name in ('colliding_predators84', 'cleanup64', 'synthetic32', 'pacman64', 'spawn_zoo', 'portal_zoo'):
        mod = importlib.import_module('moog_b200.configs.' + name)
        cfg = mod.get_config()
        np.random.seed(4)
        states = [cfg['state_initializer']() for _ in range(3)]
        blobs.append((name, C.compile_config(cfg, states, layer_capacity=getattr(mod, 'LAYER_CAPACITY', None),
                                             reset_sampler=name == 'colliding_predators84').blob))
    assert len(blobs) > 25
    for name, blob in blobs:
        assert check(blob) == 0, name
    # corruptions of one well-formed program
    good = np.frombuffer(dict(blobs)['spawn_zoo'], dtype=np.uint8)
    hdr0 = good[:C.HDR_WORDS * 4].view('<i4')
    n_ops = int(hdr0[C.H_N_OPS])

    def corrupt(edit):
        b = good.copy()
        edit(b[:C.HDR_WORDS * 4].view('<i4'), b[C.HDR_WORDS * 4:C.HDR_WORDS * 4 + 80 * n_ops].view('<i4').reshape(n_ops, 20))
        return check(b.tobytes())

    def setw(i, v):
        return lambda h, ops: h.__setitem__(i, v)

    assert check(good.tobytes()[:-8]) != 0                                  # truncated
    assert corrupt(setw(C.H_N_RULES, n_ops + 1)) != 0                        # section beyond the ops
    assert corrupt(setw(C.H_RULES, -3)) != 0
    assert corrupt(setw(C.H_VOFF, int(hdr0[C.H_N_IPOOL]))) != 0              # voff outside ipool
    assert corrupt(setw(C.H_LAYER_OFF + 1, 10 ** 6)) != 0                    # layers not a partition of the slots
    assert corrupt(setw(C.H_N_LAYERS, 99)) != 0
    assert corrupt(setw(C.H_SHAPE_TAB, -1)) != 0
    assert corrupt(setw(C.H_N_VTX, 1)) != 0                                  # outlines beyond the vertex array
    rules = int(hdr0[C.H_RULES])
    assert corrupt(lambda h, ops: ops[rules].__setitem__(0, 9999)) != 0       # unknown op kind
    assert corrupt(lambda h, ops: ops[rules].__setitem__(2, n_ops + 5)) != 0  # ConditionalRule -> no condition op
    create = [k for k in range(n_ops) if ops_kind(good, n_ops, k) == C.R_CREATE_SPRITES][0]
    assert corrupt(lambda h, ops: ops[create].__setitem__(2, 77)) != 0        # layer id
    assert corrupt(lambda h, ops: ops[create].__setitem__(6, 10 ** 7)) != 0   # sampler table outside ipool
    vanish = [k for k in range(n_ops) if ops_kind(good, n_ops, k) == C.R_VANISH_BY_FILTER][0]
    assert corrupt(lambda h, ops: ops[vanish].__setitem__(4, 10 ** 6)) != 0   # expression start


def ops_kind(blob, n_ops, k):
    from moog_b200 import compiler as C
    return int(blob[C.HDR_WORDS * 4:C.HDR_WORDS * 4 + 80 * n_ops].view('<i4').reshape(n_ops, 20)[k, 0])
