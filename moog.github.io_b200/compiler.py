"""Config compiler: MOOG component objects -> device program + state records.

Input is the dict a MOOG config's `get_config(level)` returns (reference:
moog/environment.py:28-35).  The component objects are read by duck typing on
class name and the reference's private attribute names (`Physics._forces`,
`Collision._elasticity`, `ContactReward._layers_0`, ...), so the same compiler
accepts this repo's `moog` spec classes (production) and the reference's own
instances (parity runs on the very same config object).

Output:
  * `Program` -- the binary blob described in include/moog_b200_program.h plus
    host-side metadata (layer names, capacities, action / noise layout);
  * `pack_states` -- list of `OrderedDict[str, list[Sprite]]` -> the SoA numpy
    arrays of the per-env state record.

Nothing here touches the GPU or the oracle.
"""

import collections
import itertools
import struct

import numpy as np

from . import lambdas

# ---- constants mirrored from include/moog_b200_program.h -------------------
MAGIC = 0x474F4F4D
VERSION = 1
MAX_LAYERS = 16
MAX_VERTS = 32       # MOOG_MAX_VERTS: outlines that take part in overlap tests / collisions
MAX_OUTLINE = 128    # MOOG_MAX_OUTLINE: outlines that are only moved and drawn
MAX_SLOTS = 256
DYN_FIELDS = 6
STAT_FIELDS = 10
META_FIELDS = 3
ENVI_WORDS = 8
HDR_WORDS = 64
SF_CIRCLE = 1
SF_VEL32 = 2
SF_ANGVEL_SHIFT = 2
SF_ANG_SHIFT = 4
SF_VALIAS_SHIFT = 8      # MOOG_SF_VALIAS_SHIFT
SF_VALIAS_MASK = 0x7fffff
EI_VALIAS_NEXT = 7       # MOOG_EI_VALIAS_NEXT

(H_MAGIC, H_VERSION, H_BYTES, H_N_LAYERS, H_N_SLOTS, H_K, H_N_OPS, H_N_IPOOL,
 H_N_EXPR, H_N_ENVF, H_FORCES, H_N_FORCES, H_CORR, H_N_CORR, H_RULES,
 H_N_RULES, H_TASKS, H_N_TASKS, H_ACTIONS, H_N_ACTIONS, H_ACTION_DIM,
 H_NOISE_DIM, H_R_HEIGHT, H_R_WIDTH, H_R_AA, H_R_BG, H_R_COLORMAP,
 H_R_MODIFIER, H_R_MOD_LAYER, H_R_ENABLED) = range(30)
H_RULE_NOISE_DIM = 30
H_VOFF = 31
H_LAYER_OFF = 32
H_N_VTX = 49
H_RESET, H_N_RESET, H_N_DPOOL, H_SHAPE_TAB = 51, 52, 53, 54
H_N_META, H_META_OFF = 55, 56
H_N_METAVAR, H_METAVAR_OFF, H_METAVAR_INIT = 57, 58, 59
H_VIEWS, H_N_VIEWS = 60, 61
H_MASKS, H_N_MASKS = 62, 63
VIEW_WORDS = 8           # MOOG_VIEW_WORDS: a view table row, the words H_R_HEIGHT .. H_R_ENABLED
MAX_VIEWS = 8            # MOOG_MAX_VIEWS: PILRenderer observers per program, and SpriteMask observers
MAX_META_VARS = 16
MAX_RAY_SENSORS = 8      # RaySensor observers per program
MAX_RAYS = 256           # rays per RaySensor (include/moog_b200.h moog_ray_spec)

F_DRAG, F_KINETIC_FRICTION, F_DOWN_GRAVITY, F_GRAVITY, F_RANDOM, \
    F_DIST_LINEAR, F_DIST_SPRING, F_COLLISION, F_MAZE_WALK = range(1, 10)
C_TETHER, C_TETHER_ZIPPED, C_CONSTANT_SPEED, C_MAZE_PHYSICS = 32, 33, 34, 35
R_VANISH_ON_CONTACT, R_VANISH_BY_FILTER, R_MODIFY_ON_CONTACT, \
    R_MODIFY_SPRITES, R_COND_BEGIN, R_TIMED_BEGIN, R_KEEP_NEAR_CENTER = 64, 65, 66, 67, 68, 69, 70
R_PORTAL, R_CHANGE_LAYER, R_CREATE_SPRITES, R_TREE = 71, 72, 73, 74
R_FIXATION, R_PHASESEQ_BEGIN, R_PHASE_BEGIN, R_PHASE_END = 75, 76, 77, 78
# rule classes of the reference that keep Python-side state the tracer must not guess at
_RULES_OF_THE_REFERENCE_NOT_LOWERED = ()
T_CONTACT_REWARD, T_RESET, T_STAY_ALIVE, T_TIMEOUT = 96, 97, 98, 99
A_JOYSTICK, A_GRID, A_SET_POSITION = 128, 129, 130
SC_ALL, SC_ANY, SC_COUNT, SC_CONTACT_COUNT, SC_CONTACT_ANY_COUNT, SC_CONST, \
    SC_BINARY, SC_NOT, SC_FIRST, SC_BERNOULLI, SC_TREE = 160, 161, 162, 163, 164, 165, 166, 167, 168, 169, 170
Z_GENERATE = 192
Z_N_ATTRS, Z_SHAPE_ATTR = 14, 13
ZK_CONST, ZK_UNIFORM32, ZK_DISCRETE, ZK_DISCRETE_P = 0, 1, 2, 3
# columns of the sprite observation (MOOG_OBS_*): float32 [N, n_slots, OBS_COLS]
(OBS_X, OBS_Y, OBS_SHAPE, OBS_ANGLE, OBS_SCALE, OBS_ASPECT, OBS_C0, OBS_C1, OBS_C2, OBS_OPACITY,
 OBS_X_VEL, OBS_Y_VEL, OBS_ANGLE_VEL, OBS_MASS, OBS_LAYER, OBS_ALIVE) = range(16)
OBS_COLS = 16

FL_SYMMETRIC = 1
FL_UPDATE_ANGLE_VEL = 2
FL_APPLY_DISTANT = 4
FL_APPLY_NEARBY = 8
FL_HAS_ANCHOR = 16
FL_CONSTRAINED_LR = 32
FL_CONTROL_VELOCITY = 64
FL_SAMPLE_ONE = 128
FL_PREVENT_BACKTRACKING = 256
FL_ALLOW_WALL_BACKTRACKING = 512
FL_ONLY_TURN_AT_WALL = 1024
FL_DISJOINT = 2048
FL_FAIL_GRACEFULLY = 4096

CMAP_NONE, CMAP_HSV = 0, 1
PMOD_NONE, PMOD_FIRST_PERSON, PMOD_TORUS = 0, 1, 2

OP_DTYPE = np.dtype([('kind', '<i4'), ('flags', '<i4'), ('i', '<i4', (6,)),
                     ('p', '<f8', (6,))])
EX_DTYPE = np.dtype([('op', '<i4'), ('arg', '<i4'), ('c', '<f8')])
assert OP_DTYPE.itemsize == 80 and EX_DTYPE.itemsize == 16


class CompileError(ValueError):
    """The config uses something the accelerated path cannot express."""


def _kind(obj):
    return type(obj).__name__


def _as_list(x):
    return list(x) if isinstance(x, (list, tuple)) else [x]


class Program(object):
    """Compiled task: `blob` (bytes) + the metadata the host needs."""

    def __init__(self):
        self.layer_names = []
        self.layer_cap = []
        self.layer_off = [0]
        self.ops = []            # list of dict(kind, flags, i, p)
        self.ipool = []
        self.expr = []           # list of (op, arg, c)
        self.dpool = []          # doubles: shape table / sampler parameters of the reset sampler
        self.meta_vars = collections.OrderedDict()   # env `meta_state[key]` -> envf slot (numbers; strings as codes)
        self.meta_var_init = {}  # key -> value after meta_state_initializer()
        self.meta_var_off = -1   # envf offset of the block reserved for them
        self.strings = []        # interned strings (phase names ...): code = index + 1
        self.string_vars = set() # meta_state keys that hold strings
        self.duration_draws = [] # (rule-noise column, lo, hi) of every Phase whose duration is np.random.randint(lo, hi)
        self.rule_draws = []     # (rule object, [(kind, rule-noise column, parameter)]) of traced rules that draw
        self.meta_keys = []      # `sprite.metadata[key]` columns the callables read (lambdas.metadata_columns)
        self.meta_off = 0        # envf offset of column 0 (column k of slot s: meta_off + k * n_slots + s)
        self.z_shape_ids = {}    # device sampler: shape candidate -> index of its shape record
        self.z_shape_recs = []
        self.reset_shapes = []   # shape candidates of the reset sampler, by shape id
        self.sections = {}
        self.n_envf = 0
        self.maze_offsets = {}   # maze layer name -> envf offset of its maze record
        self.action_dim = 0
        self.action_layout = []  # (key or None, kind, offset, width)
        self.noise_dim = 0
        self.rule_noise_dim = 0
        self.K = 1
        self.layer_vcap = []     # cached-vertex capacity per sprite, per layer
        self.voff = [0]          # first cached vertex of each slot
        self.render = None       # settings of view 0 (the first PILRenderer), or None
        self.views = []          # (observers key, render dict) of every PILRenderer, in observers order
        self.masks = []          # (observers key, mask dict) of every SpriteMask, in observers order
        self.rays = []           # (observers key, ray dict) of every RaySensor, in observers order (not in the blob)
        self.state_key = None    # observers key of the RawState observer, or None
        self.blob = b''

    # -- helpers used while building --
    def layer_index(self, name):
        try:
            return self.layer_names.index(name)
        except ValueError:
            raise CompileError(
                'layer {!r} is not in the environment state (layers: {})'
                .format(name, self.layer_names))

    def add_list(self, names):
        start = len(self.ipool)
        self.ipool.extend(self.layer_index(n) for n in names)
        return start, len(names)

    def add_ints(self, ints):
        start = len(self.ipool)
        self.ipool.extend(int(v) for v in ints)
        return start

    def add_expr(self, code):
        """code: list of (op, arg, c) WITHOUT the terminator; returns start."""
        if code is None:
            return -1
        start = len(self.expr)
        self.expr.extend(code)
        self.expr.append((lambdas.X_END, 0, 0.0))
        return start

    def maze_record(self, layer):
        """envf offset of the maze record of `layer` (host_maze.maze_record)."""
        from . import host_maze
        if layer not in self.maze_offsets:
            self.layer_index(layer)
            self.maze_offsets[layer] = self.alloc_envf(host_maze.MAZE_WORDS)
        return self.maze_offsets[layer]

    def intern(self, text):
        """Code of a string the env's meta_state holds or is compared with."""
        if text not in self.strings:
            self.strings.append(text)
        return float(self.strings.index(text) + 1)

    def meta_slot(self, key):
        """envf slot of meta_state[key] (a block of MAX_META_VARS slots is reserved on first use)."""
        if key not in self.meta_vars:
            if self.meta_var_off < 0:
                self.meta_var_off = self.alloc_envf(MAX_META_VARS)
            if len(self.meta_vars) >= MAX_META_VARS:
                raise CompileError('at most {} meta_state entries are carried on the device'.format(MAX_META_VARS))
            self.meta_vars[key] = self.meta_var_off + len(self.meta_vars)
        return self.meta_vars[key]

    def alloc_envf(self, n):
        start = self.n_envf
        self.n_envf += n
        return start

    def emit(self, kind, flags=0, i=(), p=()):
        i = list(i) + [0] * (6 - len(i))
        p = list(p) + [0.0] * (6 - len(p))
        self.ops.append(dict(kind=kind, flags=flags, i=i, p=p))
        return len(self.ops) - 1

    @property
    def n_slots(self):
        return self.layer_off[-1]

    @property
    def n_layers(self):
        return len(self.layer_names)

    @property
    def n_vtx(self):
        return self.voff[-1]

    def meta_values(self):
        """The meta_state variables right after meta_state_initializer() (0 for keys only rules create)."""
        out = []
        for key in self.meta_vars:
            v = self.meta_var_init.get(key, 0.0)
            out.append(self.intern(v) if isinstance(v, str) else float(v))
        return out

    def finalize(self):
        hdr = np.zeros(HDR_WORDS, dtype='<i4')
        hdr[H_VOFF] = self.add_ints(self.voff)
        hdr[H_N_VTX] = self.voff[-1]
        if len(self.views) > 1:
            # views 1..: the view table behind everything else in ipool (a program with one renderer
            # has no table, and its blob is what it was before views existed)
            hdr[H_VIEWS] = self.add_ints(w for _, r in self.views[1:] for w in _view_words(r))
            hdr[H_N_VIEWS] = len(self.views) - 1
        if self.masks:
            # the mask table behind the view table (a program without a mask has none)
            hdr[H_MASKS] = self.add_ints(w for _, m in self.masks for w in _view_words(m))
            hdr[H_N_MASKS] = len(self.masks)
        ops = np.zeros(len(self.ops), dtype=OP_DTYPE)
        for k, o in enumerate(self.ops):
            ops[k]['kind'] = o['kind']
            ops[k]['flags'] = o['flags']
            ops[k]['i'] = o['i']
            ops[k]['p'] = o['p']
        ipool = list(self.ipool)
        if len(ipool) % 2:
            ipool.append(0)
        ipool = np.array(ipool, dtype='<i4')
        expr = np.zeros(len(self.expr), dtype=EX_DTYPE)
        for k, (op, arg, c) in enumerate(self.expr):
            expr[k] = (op, arg, c)
        hdr[H_MAGIC] = MAGIC
        hdr[H_VERSION] = VERSION
        hdr[H_N_LAYERS] = self.n_layers
        hdr[H_N_SLOTS] = self.n_slots
        hdr[H_K] = self.K
        hdr[H_N_OPS] = len(ops)
        hdr[H_N_IPOOL] = len(self.ipool)
        hdr[H_N_EXPR] = len(expr)
        hdr[H_N_ENVF] = max(self.n_envf, 1)
        for name, (hs, hn) in (('forces', (H_FORCES, H_N_FORCES)),
                               ('corr', (H_CORR, H_N_CORR)),
                               ('rules', (H_RULES, H_N_RULES)),
                               ('tasks', (H_TASKS, H_N_TASKS)),
                               ('actions', (H_ACTIONS, H_N_ACTIONS))):
            start, count = self.sections.get(name, (0, 0))
            hdr[hs] = start
            hdr[hn] = count
        hdr[H_ACTION_DIM] = max(self.action_dim, 1)
        hdr[H_NOISE_DIM] = self.noise_dim
        hdr[H_RULE_NOISE_DIM] = self.rule_noise_dim
        if self.render is not None:
            hdr[H_R_HEIGHT:H_R_ENABLED + 1] = _view_words(self.render)
        hdr[H_LAYER_OFF:H_LAYER_OFF + len(self.layer_off)] = self.layer_off
        start, count = self.sections.get('reset', (0, 0))
        hdr[H_RESET], hdr[H_N_RESET] = start, count
        hdr[H_N_DPOOL] = len(self.dpool)
        hdr[H_SHAPE_TAB] = getattr(self, 'shape_tab', 0)
        hdr[H_N_META] = len(self.meta_keys)
        hdr[H_META_OFF] = self.meta_off
        if self.meta_vars:
            hdr[H_N_METAVAR] = len(self.meta_vars)
            hdr[H_METAVAR_OFF] = self.meta_var_off
            hdr[H_METAVAR_INIT] = len(self.dpool)
            self.dpool.extend(self.meta_values())
            hdr[H_N_DPOOL] = len(self.dpool)
        dpool = np.array(self.dpool, dtype='<f8')
        blob = hdr.tobytes() + ops.tobytes() + ipool.tobytes() + expr.tobytes() + dpool.tobytes()
        hdr[H_BYTES] = len(blob)
        self.blob = hdr.tobytes() + blob[HDR_WORDS * 4:]
        self.header = hdr
        return self


# ---------------------------------------------------------------------------
# physics
# ---------------------------------------------------------------------------

def _force_fn_params(fn):
    """Parameters of a DistanceForce force_fn: this repo's callable objects,
    or the reference's closures (distance_fn_force.py:48-89)."""
    kind = getattr(fn, 'kind', None)
    if kind == 'linear':
        return 'linear', (fn.zero_intercept, fn.slope, fn.event_horizon,
                          fn.apply_distant_force, fn.apply_nearby_force)
    if kind == 'spring':
        return 'spring', (fn.spring_constant, fn.equilibrium)
    cells = lambdas.closure_vars(fn)
    if {'zero_intercept', 'slope', 'event_horizon'} <= set(cells):
        return 'linear', (cells['zero_intercept'], cells['slope'],
                          cells['event_horizon'],
                          cells['apply_distant_force'],
                          cells['apply_nearby_force'])
    if {'spring_constant', 'equilibrium'} <= set(cells):
        return 'spring', (cells['spring_constant'], cells['equilibrium'])
    raise CompileError(
        'DistanceForce force_fn {!r} is not linear_force_fn / spring_force_fn; '
        'arbitrary Python force functions cannot run on the device'.format(fn))


def _emit_force(prog, force, layers):
    k = _kind(force)
    la = prog.layer_index(layers[0])
    lb = prog.layer_index(layers[1]) if len(layers) > 1 else -1
    arity = {'Drag': 1, 'KineticFriction': 1, 'DownGravity': 1,
             'RandomForce': 1, 'Gravity': 2, 'DistanceForce': 2,
             'Collision': 2, 'RandomMazeWalk': 1}.get(k)
    if arity is None:
        raise CompileError('unsupported force {}'.format(k))
    if arity != len(layers):
        raise CompileError('{} takes {} layer argument(s), got {}'.format(
            k, arity, len(layers)))
    if k == 'Drag':
        prog.emit(F_DRAG, 0, (la, -1), (force._coeff_friction,))
    elif k == 'KineticFriction':
        prog.emit(F_KINETIC_FRICTION, 0, (la, -1), (force._coeff_friction,))
    elif k == 'DownGravity':
        prog.emit(F_DOWN_GRAVITY, 0, (la, -1), (force._g,))
    elif k == 'RandomForce':
        col = prog.noise_dim
        prog.noise_dim += 2 * prog.layer_cap[la]
        prog.emit(F_RANDOM, 0, (la, -1, col), (force._max_force_magnitude,))
    elif k == 'RandomMazeWalk':
        # maze_walk.py:97-196; np.random.rand(2, 2) -> 4 noise columns per sprite
        col = prog.noise_dim
        prog.noise_dim += 4 * prog.layer_cap[la]
        fl = (FL_PREVENT_BACKTRACKING if force._prevent_backtracking else 0) | (
            FL_ALLOW_WALL_BACKTRACKING if force._allow_wall_backtracking else 0) | (
            FL_ONLY_TURN_AT_WALL if force._only_turn_at_wall else 0)
        prog.emit(F_MAZE_WALK, fl,
                  (la, -1, col, prog.maze_record(force._maze_layer)),
                  (float(force._speed),))
    elif k == 'Gravity':
        prog.emit(F_GRAVITY, FL_SYMMETRIC if force._symmetric else 0,
                  (la, lb), (force._g,))
    elif k == 'DistanceForce':
        fl = FL_SYMMETRIC if force._symmetric else 0
        kind, params = _force_fn_params(force._force_fn)
        if kind == 'linear':
            zi, slope, horizon, far, near = params
            fl |= (FL_APPLY_DISTANT if far else 0) | (
                FL_APPLY_NEARBY if near else 0)
            prog.emit(F_DIST_LINEAR, fl, (la, lb), (zi, slope, horizon))
        else:
            prog.emit(F_DIST_SPRING, fl, (la, lb), params)
    elif k == 'Collision':
        fl = (FL_SYMMETRIC if force._symmetric else 0) | (
            FL_UPDATE_ANGLE_VEL if force._update_angle_vel else 0)
        prog.emit(F_COLLISION, fl, (la, lb, int(force._max_recursion_depth)),
                  (force._elasticity,))


def _compile_physics(prog, physics):
    k = _kind(physics)
    if k != 'Physics':
        raise CompileError(
            'physics must be a Physics instance, got {}'.format(k))
    prog.K = int(physics._updates_per_env_step)
    start = len(prog.ops)
    for entry in physics._forces:
        force, args = entry[0], entry[1:]
        # physics.py:92-108: product over the layer-name lists, in order.
        for combo in itertools.product(*[_as_list(a) for a in args]):
            _emit_force(prog, force, combo)
    prog.sections['forces'] = (start, len(prog.ops) - start)

    start = len(prog.ops)
    for cp in physics._corrective_physics:
        ck = _kind(cp)
        if ck in ('Tether', 'TetherZippedLayers'):
            ls, ln = prog.add_list(cp._layer_names)
            fl = FL_UPDATE_ANGLE_VEL if cp._update_angle_vel else 0
            ax = ay = 0.0
            if cp._anchor is not None:
                fl |= FL_HAS_ANCHOR
                ax, ay = float(cp._anchor[0]), float(cp._anchor[1])
            prog.emit(C_TETHER if ck == 'Tether' else C_TETHER_ZIPPED, fl,
                      (ls, ln), (ax, ay))
        elif ck == 'ConstantSpeed':
            ls, ln = prog.add_list(cp._layer_names)
            prog.emit(C_CONSTANT_SPEED, 0, (ls, ln), (cp._speed,))
        elif ck == 'MazePhysics':
            # maze_physics.py:19-211 (its own updates_per_env_step must be 1)
            if prog.K != 1:
                raise CompileError('MazePhysics needs updates_per_env_step == 1 (maze_physics.py:207-208)')
            ls, ln = prog.add_list(list(cp._avatar_layers))
            none = float('nan')
            prog.emit(C_MAZE_PHYSICS, 0, (ls, ln, prog.maze_record(cp._maze_layer)),
                      (none if cp._constant_speed is None else float(cp._constant_speed),
                       none if cp._max_speed is None else float(cp._max_speed)))
        else:
            raise CompileError(
                'corrective physics {} is not on the accelerated path'
                .format(ck))
    prog.sections['corr'] = (start, len(prog.ops) - start)


# ---------------------------------------------------------------------------
# tasks
# ---------------------------------------------------------------------------

def _emit_condition(prog, cond):
    """State condition -> index of a MOOG_SC_* op (appended out of section)."""
    spec = lambdas.compile_state_condition(cond, prog)
    return spec


def _compile_task(prog, task, out):
    k = _kind(task)
    if k == 'CompositeTask':
        timeout = task._timeout_steps
        if np.isfinite(timeout):
            out.append(dict(kind=T_TIMEOUT, p=(float(timeout),)))
        for sub in task._tasks:
            _compile_task(prog, sub, out)
    elif k == 'StayAlive':
        out.append(dict(kind=T_STAY_ALIVE,
                        p=(float(task._reward_period),
                           float(task._reward_value))))
    elif k == 'ContactReward':
        reward, reward_code = lambdas.pair_reward(task._reward_fn)
        cond = lambdas.compile_pair_condition(task._condition)
        l0s, l0n = prog.add_list(_as_list(task._layers_0))
        l1s, l1n = prog.add_list(_as_list(task._layers_1))
        out.append(dict(
            kind=T_CONTACT_REWARD,
            i=(l0s, l0n, l1s, l1n, prog.add_expr(cond), prog.alloc_envf(1)),
            p=(float(reward), float(task._reset_steps_after_contact),
               float(prog.add_expr(reward_code) + 1) if reward_code is not None else 0.0)))
    elif k == 'Reset':
        reward, reward_op = lambdas.state_reward(task._reward_fn, prog)
        out.append(dict(
            kind=T_RESET, cond=task._condition,
            i=[0, 0 if reward_op is None else reward_op + 1, 0, 0, 0, prog.alloc_envf(1)],
            p=(float(task._steps_after_condition), float(reward))))
    else:
        raise CompileError('unsupported task {}'.format(k))


def _compile_tasks(prog, task):
    specs = []
    _compile_task(prog, task, specs)
    # Conditions are emitted first (outside any section) so that the task ops
    # themselves stay contiguous.
    for s in specs:
        if 'cond' in s:
            s['i'][0] = _emit_condition(prog, s.pop('cond'))
    start = len(prog.ops)
    for s in specs:
        prog.emit(s['kind'], 0, s.get('i', ()), s.get('p', ()))
    prog.sections['tasks'] = (start, len(prog.ops) - start)


# ---------------------------------------------------------------------------
# action spaces
# ---------------------------------------------------------------------------

def _compile_action(prog, space, key, out):
    k = _kind(space)
    if k == 'Composite':
        for sub_key, sub in space.action_spaces.items():
            _compile_action(prog, sub, sub_key, out)
        return
    ls, ln = prog.add_list(_as_list(space._action_layers))
    off = prog.action_dim
    if k == 'Joystick':
        fl = (FL_CONSTRAINED_LR if space._constrained_lr else 0) | (
            FL_CONTROL_VELOCITY if space._control_velocity else 0)
        out.append(dict(kind=A_JOYSTICK, flags=fl,
                        i=(ls, ln, off, 0, 0, prog.alloc_envf(2)),
                        p=(float(space._scaling_factor),
                           float(space._momentum))))
        width = 2
    elif k == 'Grid':
        fl = FL_CONTROL_VELOCITY if space._control_velocity else 0
        out.append(dict(kind=A_GRID, flags=fl,
                        i=(ls, ln, off, 0, 0, prog.alloc_envf(2)),
                        p=(float(space._scaling_factor),
                           float(space._momentum))))
        width = 1
    elif k == 'SetPosition':
        out.append(dict(kind=A_SET_POSITION, flags=0, i=(ls, ln, off),
                        p=(float(space._inertia),)))
        width = 2
    else:
        raise CompileError('unsupported action space {}'.format(k))
    prog.action_layout.append((key, k, off, width))
    prog.action_dim += width


def _compile_actions(prog, action_space):
    specs = []
    _compile_action(prog, action_space, None, specs)
    start = len(prog.ops)
    for s in specs:
        prog.emit(s['kind'], s['flags'], s['i'], s['p'])
    prog.sections['actions'] = (start, len(prog.ops) - start)


# ---------------------------------------------------------------------------
# rules
# ---------------------------------------------------------------------------

MAX_COND_DEPTH = 4   # MOOG_MAX_COND_DEPTH (csrc/moog_step.cu rules_step: explicit block stack)
CREATE_HEADROOM = 16  # default room for the sprites CreateSprites makes (compile_config)


def _rule_specs(prog, rule, out, depth=0):
    k = _kind(rule)
    if k in ('ConditionalRule', 'TimedRule', 'DelayedRule', 'TemporaryRule') and depth >= MAX_COND_DEPTH:
        raise CompileError('conditional / timed rules nested deeper than {} are not on the accelerated '
                           'path'.format(MAX_COND_DEPTH))
    if k == 'VanishOnContact':
        gci = rule._get_contact_indices
        l0, l1 = lambdas.contact_layers(gci)
        out.append(dict(kind=R_VANISH_ON_CONTACT,
                        i=(prog.layer_index(l0), prog.layer_index(l1))))
    elif k == 'VanishByFilter':
        code = lambdas.compile_sprite_predicate(rule._filter_fn)
        out.append(dict(kind=R_VANISH_BY_FILTER,
                        i=(prog.layer_index(rule._layer), 0,
                           prog.add_expr(code))))
    elif k == 'ModifyOnContact':
        l0s, l0n = prog.add_list(_as_list(rule._layers_0))
        l1s, l1n = prog.add_list(_as_list(rule._layers_1))
        quad = []
        for mod, filt in ((rule._modifier_0, rule._filter_0),
                          (rule._modifier_1, rule._filter_1)):
            quad.append(prog.add_expr(lambdas.compile_modifier(mod))
                        if mod is not None else -1)
            quad.append(prog.add_expr(lambdas.compile_sprite_predicate(filt)))
        out.append(dict(kind=R_MODIFY_ON_CONTACT,
                        i=(l0s, l0n, l1s, l1n, prog.add_ints(quad))))
    elif k == 'ModifySprites':
        ls, ln = prog.add_list(_as_list(rule._layers))
        mod = prog.add_expr(lambdas.compile_modifier(rule._modifier))
        filt = (prog.add_expr(lambdas.compile_sprite_predicate(rule._filter_fn))
                if rule._filter_fn else -1)
        col = 0
        if rule._sample_one:
            col = prog.rule_noise_dim
            prog.rule_noise_dim += 1
        out.append(dict(kind=R_MODIFY_SPRITES,
                        flags=FL_SAMPLE_ONE if rule._sample_one else 0,
                        i=(ls, ln, mod, filt, col)))
    elif k == 'ConditionalRule':
        sub = []
        for r in rule._rules:
            _rule_specs(prog, r, sub, depth + 1)
        out.append(dict(kind=R_COND_BEGIN, cond=rule._condition,
                        i=[0, len(sub)]))
        out.extend(sub)
    elif k in ('TimedRule', 'DelayedRule', 'TemporaryRule'):
        # timing.py:15-107; a random interval (user callable) cannot be lowered
        # (sampling the callable a few times would misclassify one that picks among few values;
        # it is called with every module-level random draw refused instead)
        try:
            with lambdas.no_randomness('{} step interval'.format(k)):
                draws = [tuple(float(v) for v in rule._step_interval()) for _ in range(2)]
        except lambdas.ImpureCallable:
            raise CompileError('{} with a random step interval is not on the accelerated path'.format(k))
        if len(set(draws)) != 1:
            raise CompileError('{} with a varying step interval is not on the accelerated path'.format(k))
        sub = []
        for r in rule._rules:
            _rule_specs(prog, r, sub, depth + 1)
        out.append(dict(kind=R_TIMED_BEGIN, i=[0, len(sub), prog.alloc_envf(2)], p=draws[0]))
        out.extend(sub)
    elif k == 'Portal':
        out.append(dict(kind=R_PORTAL, i=(prog.layer_index(rule._teleporting_layer),
                                          prog.layer_index(rule._portal_layer))))
    elif k == 'ChangeLayer':
        code = lambdas.compile_sprite_predicate(rule._filter_fn)
        out.append(dict(kind=R_CHANGE_LAYER, i=(prog.layer_index(rule._old_layer), prog.layer_index(rule._new_layer),
                                                prog.add_expr(code))))
    elif k == 'Fixation':
        out.append(dict(kind=R_FIXATION, i=(prog.layer_index(rule._agent_layer), prog.layer_index(rule._fixation_layer),
                                            prog.meta_slot(rule._meta_state_fixation_key)),
                        p=(float(rule._fixation_threshold),)))
    elif k == 'Phase':
        _phase_specs(prog, rule, out, depth, seq=-1, index=0)
    elif k == 'PhaseSequence':
        phases = list(rule._phases)
        if not phases or any(_kind(ph) != 'Phase' for ph in phases):
            raise CompileError('PhaseSequence takes Phase instances')
        seq = prog.alloc_envf(2)          # current phase index, its value when the pass began
        name_slot = prog.meta_slot(rule._meta_state_key) if rule._meta_state_key is not None else -1
        if rule._meta_state_key is not None:
            prog.string_vars.add(rule._meta_state_key)
        names = len(prog.dpool)
        prog.dpool.extend(prog.intern(ph.name) for ph in phases)
        out.append(dict(kind=R_PHASESEQ_BEGIN, i=(seq, len(phases), name_slot, 0, names)))
        for index, ph in enumerate(phases):
            _phase_specs(prog, ph, out, depth, seq=seq, index=index, name_slot=name_slot, names=names, n_phases=len(phases))
    elif k == 'CreateSprites':
        # create_sprites.py:27-34; the generator's recipe is sampled on the device (Philox), like a reset group
        gen = _Recipe(rule._generator)
        count, lo, hi, col = gen.num_sprites, 0.0, 0.0, 0.0
        if callable(gen.num_sprites):
            # num_sprites=lambda: np.random.randint(lo, hi): drawn per call from a rule-noise column of its own
            drawn = lambdas.randint_range(gen.num_sprites)
            if drawn is None:
                raise CompileError('CreateSprites with a random number of sprites per call is only lowered when it is '
                                   '`np.random.randint(lo, hi)`')
            count, lo, hi, col = drawn[1] - 1, float(drawn[0]), float(drawn[1]), float(prog.rule_noise_dim)
            prog.rule_noise_dim += 1
        lay = prog.layer_index(rule._layer)
        table, meta_flags, ext = _sampler_group(prog, gen.factor_dist, lay)
        t_start = _emit_sampler_table(prog, table, ext)
        ls, ln = prog.add_list(_as_list(rule._without_overlapping))
        out.append(dict(kind=R_CREATE_SPRITES, flags=FL_FAIL_GRACEFULLY if gen.fail_gracefully else 0,
                        i=(lay, int(count), ls, ln, t_start, meta_flags),
                        p=(float(gen.max_recursion_depth), lo, hi, col)))
    elif k == 'KeepNearCenter':
        layers = list(rule._layers_to_center)
        ls, ln = prog.add_list(layers)
        grid = rule._grid_cell
        out.append(dict(kind=R_KEEP_NEAR_CENTER, i=(prog.layer_index(rule._agent_layer), ls, ln),
                        p=(float(grid[0]), float(grid[1]))))
    elif callable(getattr(type(rule), 'step', None)) and k not in _RULES_OF_THE_REFERENCE_NOT_LOWERED:
        # a rule class of the config's own (functional_maze.py:18-67): its step() is traced path by path
        try:
            start, count, base, initial = lambdas.trace_rule(rule, prog)
        except lambdas.LoweringError as exc:
            raise CompileError('game rule {} is not on the accelerated path and cannot be traced: {}'.format(k, exc))
        first = len(prog.dpool)
        prog.dpool.extend(float(v) for v in initial)
        out.append(dict(kind=R_TREE, i=(start, count, base, len(initial), first)))
    else:
        raise CompileError(
            'game rule {} is not on the accelerated path'.format(k))


def _phase_specs(prog, phase, out, depth, seq, index, name_slot=-1, names=0, n_phases=0):
    """task_phases.py:18-95: MOOG_R_PHASE_BEGIN, [a MOOG_R_COND_BEGIN on `step_count == 0` around the
    one-time rules], the continual rules, MOOG_R_PHASE_END."""
    if depth + 2 > MAX_COND_DEPTH:
        raise CompileError('phases nested deeper than {} blocks are not on the accelerated path'.format(MAX_COND_DEPTH))
    base = prog.alloc_envf(3)             # should_end, step_count, duration
    duration = phase._duration
    drawn = lambdas.randint_range(duration) if callable(duration) else None
    col, fixed, lo, hi = 0, 0.0, 0.0, 0.0
    if drawn is not None:
        lo, hi = float(drawn[0]), float(drawn[1])
        col = prog.rule_noise_dim
        prog.rule_noise_dim += 1
        prog.duration_draws.append((col, drawn[0], drawn[1]))
    else:
        try:
            with lambdas.no_randomness('Phase duration'):
                fixed = float(duration() if callable(duration) else duration)
        except lambdas.ImpureCallable:
            raise CompileError('a random Phase duration is only lowered when it is `np.random.randint(lo, hi)`')
    once, always = [], []
    for r in phase._one_time_rules:
        _rule_specs(prog, r, once, depth + 2)
    for r in phase._continual_rules:
        _rule_specs(prog, r, always, depth + 1)
    block = []
    if once:
        first = prog.add_expr([(lambdas.X_ENVF, base + 1, 0.0), (lambdas.X_CONST, 0, 0.0), (lambdas.X_EQ, 0, 0.0)])
        first_op = prog.emit(SC_TREE, 0, (prog.add_ints([0, first, -1, 0, -1, 0, 0, 0]), 1))
        block.append(dict(kind=R_COND_BEGIN, i=[first_op, len(once)]))
        block += once
    block += always
    end = lambdas._unwrap(phase._end_condition, 'end_condition')  # pylint: disable=protected-access
    never = False
    try:
        never = end(None, None) is False
    except Exception:  # pylint: disable=broad-except
        never = False
    block.append(dict(kind=R_PHASE_END, i=[-1, base, seq, name_slot, names, n_phases], p=(float(index),),
                      **({} if never else {'cond': end})))
    out.append(dict(kind=R_PHASE_BEGIN, i=(seq, len(block), index, base, col), p=(fixed, lo, hi)))
    out.extend(block)


def _layer_moves(rules):
    """(old_layer, new_layer) of every ChangeLayer rule, nested ones included."""
    out = []
    for r in (rules or ()):
        k = _kind(r)
        if k == 'ChangeLayer':
            out.append((r._old_layer, r._new_layer))
        elif hasattr(r, '_rules'):
            out += _layer_moves(r._rules)
    return out


def _created(rules):
    """(layer, generator) of every CreateSprites rule, nested ones included."""
    out = []
    for r in (rules or ()):
        if _kind(r) == 'CreateSprites':
            out.append((r._layer, r._generator))
        elif hasattr(r, '_rules'):
            out += _created(r._rules)
    return out


class _Recipe(object):
    """What a generate_sprites closure was made with (sprite_generators.py:26-29)."""

    def __init__(self, gen):
        names = ('factor_dist', 'num_sprites', 'max_recursion_depth', 'fail_gracefully')
        if all(hasattr(gen, n) for n in names):          # this repo's generate_sprites says so itself
            values = {n: getattr(gen, n) for n in names}
        else:                                            # the reference's: the closure's free variables
            values = lambdas.closure_vars(gen) if callable(gen) else {}
        if any(n not in values for n in names):
            raise CompileError('CreateSprites needs a generator made by sprite_generators.generate_sprites')
        self.factor_dist = values['factor_dist']
        self.num_sprites = values['num_sprites']
        self.max_recursion_depth = values['max_recursion_depth']
        self.fail_gracefully = bool(values['fail_gracefully'])


def _generator_outline(gen):
    """Most vertices a sprite drawn from the generator's factor distribution can have."""
    from moog import sprite as sprite_lib
    flat, _ = _lower_distribution(gen.factor_dist)
    leaf = flat.get('shape', ('discrete', [_sprite_defaults()['shape']]))
    if leaf[0] not in ('discrete', 'discrete_p'):
        raise CompileError('the shape must be a plain Discrete / constant factor on the device sampler')
    return max(len(sprite_lib.Sprite(x=0., y=0., shape=shape).vertices) for shape in leaf[1])


def _compile_rules(prog, rules):
    specs = []
    for r in (rules or ()):
        _rule_specs(prog, r, specs)
    for s in specs:
        if 'cond' in s:
            s['i'][0] = _emit_condition(prog, s.pop('cond'))
    start = len(prog.ops)
    for s in specs:
        prog.emit(s['kind'], s.get('flags', 0), s.get('i', ()), s.get('p', ()))
    prog.sections['rules'] = (start, len(prog.ops) - start)


# ---------------------------------------------------------------------------
# observers
# ---------------------------------------------------------------------------

def _view_words(r):
    """The MOOG_VIEW_WORDS settings of one renderer (header words H_R_HEIGHT .. H_R_ENABLED)."""
    bg = r['bg']
    return [r['height'], r['width'], r['aa'], int(bg[0]) | (int(bg[1]) << 8) | (int(bg[2]) << 16),
            r['colormap'], r['modifier'], r['modifier_layer'], 1]


def _compile_render(prog, observers):
    prog.state_key = None
    prog.views = []
    prog.masks = []
    prog.rays = []
    for key, obs in (observers or {}).items():
        if _kind(obs) == 'PILRenderer':
            if len(prog.views) >= MAX_VIEWS:
                raise CompileError('at most {} PILRenderer observers are supported'.format(MAX_VIEWS))
            prog.views.append((key, _lower_renderer(prog, obs)))
        elif _kind(obs) == 'SpriteMask':
            if len(prog.masks) >= MAX_VIEWS:
                raise CompileError('at most {} SpriteMask observers are supported'.format(MAX_VIEWS))
            prog.masks.append((key, _lower_mask(prog, obs)))
        elif _kind(obs) == 'RaySensor':
            if len(prog.rays) >= MAX_RAY_SENSORS:
                raise CompileError('observer {!r}: at most {} RaySensor observers are supported'.format(
                    key, MAX_RAY_SENSORS))
            prog.rays.append((key, _lower_rays(prog, key, obs)))
        elif _kind(obs) == 'RawState':
            if prog.state_key is not None:
                raise CompileError('only one RawState observer is supported')
            prog.state_key = key
        elif callable(obs) and _kind(obs) == 'function':
            continue  # e.g. runtime_benchmark's `lambda _: None`
        else:
            raise CompileError('unsupported observer {}'.format(_kind(obs)))
    prog.render = prog.views[0][1] if prog.views else None


def _lower_renderer(prog, renderer):
    size = tuple(renderer._image_size)
    if len(size) != 2:
        raise CompileError('image_size must be (height, width)')
    bg = getattr(renderer, '_bg_color', None)
    if bg is None:
        bg = renderer._canvas_bg.getpixel((0, 0))
    fn = renderer.color_to_rgb
    if fn is None:
        cmap = CMAP_NONE
    elif getattr(fn, '__name__', '') == 'hsv_to_rgb':
        cmap = CMAP_HSV
    else:
        probe = (3, 5, 7)
        try:
            same = tuple(fn(probe)) == probe
        except Exception:  # pylint: disable=broad-except
            same = False
        if not same:
            raise CompileError(
                'color_to_rgb must be None or "hsv_to_rgb" on the device path')
        cmap = CMAP_NONE
    modifier, mod_layer = _lower_modifier(prog, renderer._polygon_modifier)
    # pil_renderer.py:46,65-66: canvas = (aa*size[0], aa*size[1]) is handed to
    # PIL as (width, height) while the array that comes back is [height, width].
    return dict(height=int(size[1]), width=int(size[0]),
                aa=int(renderer._anti_aliasing), bg=tuple(bg)[:3],
                colormap=cmap, modifier=modifier,
                modifier_layer=mod_layer)


def _lower_modifier(prog, pm):
    """(MOOG_PMOD_*, agent layer) of a polygon modifier."""
    pk = _kind(pm)
    if pk == 'FirstPersonAgent':
        return PMOD_FIRST_PERSON, prog.layer_index(pm._agent_layer)
    if pk == 'TorusGeometry':
        return PMOD_TORUS, 0
    if pk != 'DoNothing':
        raise CompileError('unsupported polygon modifier {}'.format(pk))
    return PMOD_NONE, 0


def _lower_mask(prog, mask):
    """A SpriteMask as a view row: anti_aliasing 1, no background, no colour map."""
    size = tuple(mask._image_size)
    if len(size) != 2:
        raise CompileError('image_size must be (width, height)')
    modifier, mod_layer = _lower_modifier(prog, mask._polygon_modifier)
    return dict(height=int(size[1]), width=int(size[0]), aa=1, bg=(0, 0, 0), colormap=CMAP_NONE,
                modifier=modifier, modifier_layer=mod_layer)


def _lower_rays(prog, key, sensor):
    """A RaySensor as the fields of include/moog_b200.h moog_ray_spec, its direction table included."""
    def bad(what):
        return CompileError('observer {!r}: RaySensor {}'.format(key, what))
    names = [sensor._agent_layer] + list(prog.layer_names if sensor._layers is None else sensor._layers)
    for name in names:
        if name not in prog.layer_names:
            raise bad('names layer {!r}, which is not in the environment state (layers: {})'.format(
                name, prog.layer_names))
    R = sensor._num_rays
    if isinstance(R, bool) or not isinstance(R, (int, np.integer)) or not 1 <= R <= MAX_RAYS:
        raise bad('num_rays must be an integer in [1, {}], not {!r}'.format(MAX_RAYS, R))
    max_range, fov = float(sensor._max_range), float(sensor._fov)
    if not (np.isfinite(max_range) and max_range > 0):
        raise bad('max_range must be finite and > 0, not {!r}'.format(sensor._max_range))
    if not 0 < fov <= 2 * np.pi:
        raise bad('fov must be in (0, 2 pi], not {!r}'.format(sensor._fov))
    index = sensor._agent_index
    if isinstance(index, bool) or not isinstance(index, (int, np.integer)) or index < 0:
        raise bad('agent_index must be an integer >= 0, not {!r}'.format(index))
    layers = 0
    for name in names[1:]:
        layers |= 1 << prog.layer_index(name)
    return dict(agent_layer=prog.layer_index(names[0]), agent_index=int(index), layers=layers,
                num_rays=int(R), max_range=max_range,
                dirs=np.ascontiguousarray(sensor.directions(), dtype=np.float64))


# ---------------------------------------------------------------------------
# entry points
# ---------------------------------------------------------------------------

def compile_config(config, sample_states, layer_capacity=None, reset_sampler=False):
    """Compile a MOOG config dict.

    Args:
        config: dict with the reference's Environment kwargs
            (environment.py:28-35).
        sample_states: list of states (`OrderedDict[str, list[Sprite]]`) from
            the config's state_initializer; fixes layer names / order and the
            per-layer capacities (max count seen).
        layer_capacity: optional {layer: capacity} overrides.
    """
    prog = Program()
    first = sample_states[0]
    prog.layer_names = list(first.keys())
    if len(prog.layer_names) > MAX_LAYERS:
        raise CompileError('at most {} layers'.format(MAX_LAYERS))
    for st in sample_states:
        if list(st.keys()) != prog.layer_names:
            raise CompileError('state initializer changed its layer set')
    caps = [max(len(st[name]) for st in sample_states)
            for name in prog.layer_names]
    # ChangeLayer appends sprites of one layer to another (change_layer.py:34-45): the receiving layer
    # gets room for every sprite that can arrive, and slots wide enough for their outlines
    moves = _layer_moves(config.get('game_rules', ()))
    for old, new in moves:
        caps[prog.layer_names.index(new)] += caps[prog.layer_names.index(old)]
    # CreateSprites appends to a layer for as long as the episode lasts (create_sprites.py:27-34); the
    # record gives the layer room for CREATE_HEADROOM more sprites unless `layer_capacity` says how many
    # (an env whose layer is full flags MOOG_ERR_LAYER_OVERFLOW and creates nothing)
    created = [(name, _Recipe(gen)) for name, gen in _created(config.get('game_rules', ()))]
    for name in {name for name, _ in created}:
        if name not in (layer_capacity or {}):
            caps[prog.layer_names.index(name)] += CREATE_HEADROOM
    for name, cap in (layer_capacity or {}).items():
        caps[prog.layer_index(name)] = max(cap, caps[prog.layer_index(name)])
    prog.layer_cap = [int(c) for c in caps]
    prog.layer_off = [0] + [int(v) for v in np.cumsum(caps)]
    if prog.n_slots > MAX_SLOTS:
        raise CompileError('at most {} sprites per env'.format(MAX_SLOTS))
    vcap = []
    for name in prog.layer_names:
        nvs = [len(sp.vertices) for st in sample_states for sp in st[name]]
        vcap.append(max(nvs) if nvs else 0)
    if max(vcap + [0]) > MAX_OUTLINE:
        raise CompileError(
            'a sprite outline has {} vertices; the device path supports at '
            'most {}'.format(max(vcap), MAX_OUTLINE))
    for old, new in moves:
        io, in_ = prog.layer_names.index(old), prog.layer_names.index(new)
        vcap[in_] = max(vcap[in_], vcap[io])
    for name, gen in created:
        il = prog.layer_names.index(name)
        vcap[il] = max(vcap[il], _generator_outline(gen))
    prog.layer_vcap = vcap
    voff = [0]
    for cap, vc in zip(caps, vcap):
        for _ in range(cap):
            voff.append(voff[-1] + vc)
    prog.voff = voff

    meta_init = config.get('meta_state_initializer')
    meta_init = meta_init() if callable(meta_init) else meta_init
    if meta_init is not None:
        # environment.py:86: a fresh meta_state per episode.  A dict of numbers / strings becomes variables
        # of the env's record; anything else has no device form
        if not isinstance(meta_init, dict):
            raise CompileError('meta_state must be None or a dict of numbers / strings on the device path')
        for key, value in meta_init.items():
            if not (isinstance(value, (bool, int, float, str)) or hasattr(value, '__float__')):
                raise CompileError('meta_state[{!r}] = {!r}: only numbers and strings are carried on the device'.format(key, value))
            prog.meta_var_init[key] = value if isinstance(value, str) else float(value)
            prog.meta_slot(key)
    with lambdas.metadata_columns(prog.meta_keys):
        _compile_physics(prog, config['physics'])
        _compile_tasks(prog, config['task'])
        _compile_actions(prog, config['action_space'])
        _compile_rules(prog, config.get('game_rules', ()))
    _compile_render(prog, config.get('observers', {}))
    if prog.meta_keys:
        # numeric sprite.metadata[key] values travel with the sprite: one envf column of n_slots doubles per key
        prog.meta_off = prog.alloc_envf(len(prog.meta_keys) * prog.n_slots)
    if reset_sampler:
        _compile_reset_sampler(prog, config['state_initializer'])
    _finish_z_shapes(prog)
    _emit_shape_table_if_needed(prog, sample_states, bool(prog.z_shape_recs))
    _check_outline_caps(prog)
    return prog.finalize()


# ---------------------------------------------------------------------------
# device-side reset sampler (SURVEY section 8 f1)
# ---------------------------------------------------------------------------

_ATTR_KEYS = ('x', 'y', 'x_vel', 'y_vel', 'angle', 'angle_vel', 'mass', 'scale',
              'aspect_ratio', 'c0', 'c1', 'c2', 'opacity')


def _flatten_distribution(dist):
    """Product / Continuous / Discrete tree -> {key: ('uniform', lo, hi) |
    ('discrete', [values])}; anything else cannot run on the device."""
    k = _kind(dist)
    if k == 'Product':
        out = {}
        for c in dist.components:
            out.update(_flatten_distribution(c))
        return out
    if k == 'Continuous':
        if str(dist.dtype) != 'float32':
            raise CompileError('the device sampler draws float32 Continuous factors only')
        return {dist.key: ('uniform', float(dist.minval), float(dist.maxval))}
    if k == 'Discrete':
        if getattr(dist, 'probs', None) is not None:
            # distributions.py:127-129: rng.choice(n, p=probs) -- the first candidate whose cumulative
            # probability exceeds the uniform
            probs = np.asarray(dist.probs, dtype=np.float64)
            if len(probs) != len(dist.candidates) or (probs < 0).any() or not probs.sum() > 0:
                raise CompileError('Discrete: one non-negative probability per candidate expected')
            cum = np.cumsum(probs)
            return {dist.key: ('discrete_p', list(dist.candidates), [float(v) for v in cum / cum[-1]])}
        return {dist.key: ('discrete', list(dist.candidates))}
    raise CompileError(
        'factor distribution {} cannot be sampled on the device (supported: Product of '
        'Continuous / Discrete / constants); use the host pool (reset_sampler=False)'.format(k))


def _lower_distribution(dist):
    """Factor distribution -> (leaves, extensions).  `leaves` is the flat part
    ({key: leaf}, see _flatten_distribution); `extensions` are the components of the top-level
    Product that are not flat: ('mixture', [leaves of each alternative], probs) and
    ('filtered', leaves of the base, [(key, lo, hi) of the Continuous box it is tested against],
    keep_if_inside) for Selection / SetMinus (distributions.py: Mixture, SetMinus, Selection)."""
    k = _kind(dist)
    if k == 'Product':
        leaves, ext = {}, []
        for c in dist.components:
            l2, e2 = _lower_distribution(c)
            leaves.update(l2)
            ext.extend(e2)
        return leaves, ext
    if k == 'Mixture':
        alts = [_flatten_distribution(c) for c in dist.components]
        keys = set(alts[0])
        if any(set(a) != keys for a in alts):
            raise CompileError('the alternatives of a Mixture must produce the same factors')
        probs = [float(v) for v in dist.probs]
        return {}, [('mixture', alts, probs)]
    if k in ('SetMinus', 'Selection'):
        base = _flatten_distribution(dist.base)
        box = _flatten_distribution(dist.filtering if k == 'Selection' else dist.hold_out)
        if any(v[0] != 'uniform' for v in box.values()):
            raise CompileError('{} against anything but a box of Continuous factors is not on the device sampler'.format(k))
        return {}, [('filtered', base, [(key, v[1], v[2]) for key, v in box.items()], k == 'Selection')]
    if k == 'Intersection':
        # distributions.py:211-247: sample component `index_for_sampling`, reject unless every component
        # contains the sample -- for Products of Continuous factors that is one box, the intersection
        idx = int(dist.index_for_sampling)
        base = _flatten_distribution(dist.components[idx])
        lo, hi = {}, {}
        for j, c in enumerate(dist.components):
            if j == idx:
                continue
            for key, v in _flatten_distribution(c).items():
                if v[0] != 'uniform':
                    raise CompileError('Intersection with anything but boxes of Continuous factors is not on the device sampler')
                lo[key] = max(lo.get(key, -np.inf), float(v[1]))
                hi[key] = min(hi.get(key, np.inf), float(v[2]))
        return {}, [('filtered', base, [(key, lo[key], hi[key]) for key in lo], True)]
    if k == 'DependentDistribution':
        # distributions.py:420-470: some factors are a deterministic function of the sampled ones; the
        # function is traced once into expressions over the independent factors
        indep = _flatten_distribution(dist._independent_distrib)  # pylint: disable=protected-access
        codes = lambdas.compile_dependent_fn(dist._dependent_fn, list(indep), list(dist._dependent_fn_keys))  # pylint: disable=protected-access
        f32 = {key for key, v in indep.items() if v[0] == 'uniform'}
        return indep, [('dependent', {key: v for key, v in codes.items()}, f32)]
    return _flatten_distribution(dist), []


def _emit_shape_table_if_needed(prog, sample_states, reset_sampler):
    """A modifier that assigns `scale` / `aspect_ratio` makes the device re-derive the sprite's outline
    from its shape (sprite.py:411-424): the COM-centred unit outlines of every shape the sample states
    show go into the blob (shape records, MOOG_H_SHAPE_TAB), and pack_states numbers the sprites'
    shapes by that table."""
    reshaping = {lambdas.ATTRS.index(a) for a in lambdas.RESHAPING}
    needs = any(op == lambdas.X_STORE and arg in reshaping for op, arg, _ in prog.expr)
    prog.shape_table = None
    if not needs:
        return
    if reset_sampler:
        raise CompileError('rules that assign scale / aspect_ratio are not combined with the device sampler '
                           '(reset_mode=\'device\' / CreateSprites) yet')
    table = ShapeTable()
    for st in sample_states:
        for name in prog.layer_names:
            for sp in st[name]:
                table.add(sp._shape_path.vertices[:-1], getattr(sp, 'shape', None))  # pylint: disable=protected-access
    shape_off = []
    for verts, nv in zip(table.verts, table.nv):
        shape_off.append(len(prog.dpool))
        prog.dpool.extend([float(nv), 0.0, 0.0, 0.0, 0.0, 0.0] + [float(v) for v in verts[:nv].reshape(-1)])
    prog.shape_tab = prog.add_ints(shape_off)
    prog.shape_table = table
    prog.n_table_shapes = len(table.nv)


def _shape_record(shape):
    """Shape record of include/moog_b200_program.h for one shape candidate."""
    from moog import sprite as sprite_lib
    sp = sprite_lib.Sprite(x=0., y=0., shape=shape)
    base = np.asarray(sp._shape_path.vertices[:-1], dtype=np.float64)  # pylint: disable=protected-access
    if len(base) > MAX_OUTLINE:
        raise CompileError('sprite outline has {} vertices; the device path supports at most {}'.format(
            len(base), MAX_OUTLINE))
    ixy = np.asarray(sp._x_y_rotational_inertia, dtype=np.float64)  # pylint: disable=protected-access
    centroid = np.asarray(sp.position, dtype=np.float64)             # (0, 0) + raw centroid
    rec = [float(len(base)), 1.0 if (isinstance(shape, str) and shape == 'circle') else 0.0,
           float(ixy[0]), float(ixy[1]), float(centroid[0]), float(centroid[1])]
    rec += [float(v) for v in base.reshape(-1)]
    return rec


def _sprite_defaults():
    import inspect
    from moog import sprite as sprite_lib
    return {k: p.default for k, p in inspect.signature(sprite_lib.Sprite.__init__).parameters.items()
            if p.default is not inspect.Parameter.empty}


def _z_shape_id(prog, shape):
    """Index of a shape candidate in the blob's shape records (device sampler)."""
    key = shape if isinstance(shape, str) else np.asarray(shape, dtype=np.float64).tobytes()
    if key not in prog.z_shape_ids:
        prog.z_shape_ids[key] = len(prog.z_shape_recs)
        prog.z_shape_recs.append(_shape_record(shape))
        prog.reset_shapes.append(shape)
    return prog.z_shape_ids[key]


def _sampler_group(prog, factor_dist, lay):
    """One generate_sprites recipe -> (factor table, dtype flags of the sprites it makes, extension
    components) for the device sampler (reset groups and CreateSprites rules)."""
    defaults = _sprite_defaults()
    flat, extensions = _lower_distribution(factor_dist)
    table, meta_flags = [], 0
    sampled32 = set()
    for key in _ATTR_KEYS + ('shape',):
        kind, payload = 'discrete', [defaults[key]]
        cum = None
        if key in flat:
            kind, payload = flat[key][0], list(flat[key][1:]) if flat[key][0] == 'uniform' else flat[key][1]
            cum = flat[key][2] if kind == 'discrete_p' else None
        if kind == 'uniform':
            table.append((ZK_UNIFORM32, payload))
            sampled32.add(key)
        else:
            values = [_z_shape_id(prog, v) for v in payload] if key == 'shape' else [float(v) for v in payload]
            if key == 'shape':
                for sid in values:
                    if int(prog.z_shape_recs[sid][0]) > prog.layer_vcap[lay]:
                        raise CompileError(
                            'a shape candidate has {} vertices, more than the sample states showed for layer '
                            '{!r} ({}); pass more sample states'.format(
                                int(prog.z_shape_recs[sid][0]), prog.layer_names[lay], prog.layer_vcap[lay]))
            if cum is not None and len(values) > 1:
                table.append((ZK_DISCRETE_P, values + cum))
            else:
                table.append((ZK_CONST if len(values) == 1 else ZK_DISCRETE, values))
    # factors drawn by the extensions: float32 iff every alternative draws them from a Continuous
    ext_specs = []
    for comp in extensions:
        if comp[0] == 'dependent':
            deps = []
            for key, (code, reads) in comp[1].items():
                if key == 'shape':
                    raise CompileError('the shape must be a plain Discrete / constant factor on the device sampler')
                # NumPy: an expression over float32 draws and python scalars stays float32
                is32 = bool(reads) and all(_ATTR_KEYS[a] in comp[2] for a in reads)
                if is32:
                    sampled32.add(key)
                deps.append((_ATTR_KEYS.index(key), prog.add_expr(code), 1 if is32 else 0))
            ext_specs.append(dict(kind=3, deps=deps))
            continue
        groups = comp[1] if comp[0] == 'mixture' else [comp[1]]
        for key in groups[0]:
            if key == 'shape':
                raise CompileError('the shape must be a plain Discrete / constant factor on the device sampler')
            kinds = {g[key][0] for g in groups}
            if kinds == {'uniform'}:
                sampled32.add(key)
            elif key in ('x_vel', 'y_vel', 'angle', 'angle_vel') and 'uniform' in kinds:
                raise CompileError('factor {!r} is float32 in some Mixture alternatives only'.format(key))

        def enc(leaves_):
            out_ = []
            for key_, leaf in leaves_.items():
                values = list(leaf[1:]) if leaf[0] == 'uniform' else [float(v) for v in leaf[1]]
                kind_ = ZK_UNIFORM32 if leaf[0] == 'uniform' else (ZK_CONST if len(values) == 1 else ZK_DISCRETE)
                if leaf[0] == 'discrete_p' and len(values) > 1:
                    kind_, values = ZK_DISCRETE_P, values + list(leaf[2])
                out_.append((_ATTR_KEYS.index(key_), kind_, values))
            return out_
        if comp[0] == 'mixture':
            ext_specs.append(dict(kind=1, alts=[enc(a) for a in comp[1]], probs=comp[2]))
        else:
            ext_specs.append(dict(kind=2, base=enc(comp[1]), keep=bool(comp[3]),
                                  box=[(_ATTR_KEYS.index(key), lo_, hi_) for key, lo_, hi_ in comp[2]]))
    if {'x_vel', 'y_vel'} <= sampled32:
        meta_flags |= SF_VEL32
    if 'angle_vel' in sampled32:
        meta_flags |= 1 << SF_ANGVEL_SHIFT
    # (the angle is never float32 at birth: Sprite.__init__ stores float(angle), sprite.py:310)
    return table, meta_flags, ext_specs


def _emit_sampler_table(prog, table, ext):
    """Writes a group's factor table and extension program into the pools; returns the ipool start."""
    tab = []
    def count(kind, values):        # candidates of a leaf (a weighted one carries its cumulative probabilities too)
        return len(values) // 2 if kind == ZK_DISCRETE_P else len(values)

    for kind, values in table:
        tab += [kind, len(prog.dpool), count(kind, values)]
        prog.dpool.extend(float(v) for v in values)

    def put_leaves(leaves_):
        out_ = [len(leaves_)]
        for attr, kind, values in leaves_:
            out_ += [attr, kind, len(prog.dpool), count(kind, values)]
            prog.dpool.extend(float(v) for v in values)
        return out_
    # extension program: [n_ext, then per component: 1, n_alt, probs dpool index, alternatives... |
    #                     2, keep_if_inside, base leaves, n_box, (attr, dpool index of lo hi)... |
    #                     3, n, (attr, expression start, float32?)...]
    tab.append(len(ext))
    for comp in ext:
        if comp['kind'] == 3:
            tab += [3, len(comp['deps'])]
            for attr, start_, is32 in comp['deps']:
                tab += [attr, start_, is32]
        elif comp['kind'] == 1:
            cum = list(np.cumsum(comp['probs']))
            tab += [1, len(comp['alts']), len(prog.dpool)]
            prog.dpool.extend(float(v) for v in cum)
            for alt in comp['alts']:
                tab += put_leaves(alt)
        else:
            tab += [2, 1 if comp['keep'] else 0] + put_leaves(comp['base']) + [len(comp['box'])]
            for attr, lo_, hi_ in comp['box']:
                tab += [attr, len(prog.dpool)]
                prog.dpool.extend([float(lo_), float(hi_)])
    return prog.add_ints(tab)


def _finish_z_shapes(prog):
    """Shape records of every candidate shape the device sampler can draw (MOOG_H_SHAPE_TAB)."""
    if not prog.z_shape_recs:
        return
    shape_off = []
    for rec_ in prog.z_shape_recs:
        shape_off.append(len(prog.dpool))
        prog.dpool.extend(rec_)
    prog.shape_tab = prog.add_ints(shape_off)


def _compile_reset_sampler(prog, state_initializer):
    """Traces the state initializer (this repo's sprite_generators record what they
    are asked for) and lowers every generate_sprites group to a MOOG_Z_GENERATE op."""
    import inspect
    from moog import sprite as sprite_lib
    from moog.state_initialization import sprite_generators as sg
    if not hasattr(sg, 'recording'):
        raise CompileError('the device reset sampler needs this repo\'s moog.state_initialization package')
    with sg.recording() as records:
        state = state_initializer()
    if list(state.keys()) != prog.layer_names:
        raise CompileError('state initializer changed its layer set')
    slot_of, layer_of = {}, {}
    for l, name in enumerate(prog.layer_names):
        for k, sp in enumerate(state[name]):
            slot_of[id(sp)] = prog.layer_off[l] + k
            layer_of[id(sp)] = l
    specs = []
    for rec in records:
        count_range = None
        if callable(rec['num_sprites']):
            count_range = rec.get('count_range')
            if count_range is None:
                raise CompileError('a random number of generated sprites is only lowered when it is drawn as '
                                   '`np.random.randint(lo, hi)`')
            if len(rec['out']) != count_range[1] - 1:
                raise CompileError('the traced initializer produced fewer sprites than the largest count')
        elif len(rec['out']) != rec['num_sprites']:
            raise CompileError('the traced initializer produced fewer sprites than asked for')
        if not rec['out']:
            continue
        try:
            slots = [slot_of[id(s)] for s in rec['out']]
            avoid = [slot_of[id(s)] for s in rec['avoid']]
        except KeyError:
            raise CompileError('a generated or avoided sprite is not part of the returned state')
        if slots != list(range(slots[0], slots[0] + len(slots))):
            raise CompileError('the sprites of one generate_sprites call must stay together, in order, in one layer')
        if len({layer_of[id(s)] for s in rec['out']}) != 1:
            raise CompileError('the sprites of one generate_sprites call must stay in one layer')
        if any(a >= slots[0] for a in avoid):
            raise CompileError('generated sprites can only avoid sprites in earlier slots')
        lay = layer_of[id(rec['out'][0])]
        if slots[0] + len(slots) != prog.layer_off[lay] + len(state[prog.layer_names[lay]]):
            raise CompileError('generated sprites must be the last sprites of their layer')
        table, meta_flags, ext_specs = _sampler_group(prog, rec['factor_dist'], lay)
        specs.append(dict(first=slots[0], count=len(slots), count_range=count_range, avoid=avoid, table=table,
                          meta_flags=meta_flags, ext=ext_specs,
                          flags=(FL_DISJOINT if rec['disjoint'] else 0) | (
                              FL_FAIL_GRACEFULLY if rec['fail_gracefully'] else 0),
                          max_depth=float(rec['max_recursion_depth'])))
    if not specs:
        raise CompileError('the state initializer never called generate_sprites: nothing to sample on the device')
    for sp_ in specs:      # a group of random size leaves the rest of its layer's slots empty: it must be the last one
        if sp_['count_range']:
            lay_ = max(l for l in range(prog.n_layers) if prog.layer_off[l] <= sp_['first'])
            if any(o is not sp_ and sp_['first'] < o['first'] < prog.layer_off[lay_ + 1] for o in specs):
                raise CompileError('a generate_sprites group with a random number of sprites must be the last one of its layer')
    emitted = []
    for sp_ in specs:
        a_start = prog.add_ints(sp_['avoid'])
        t_start = _emit_sampler_table(prog, sp_['table'], sp_['ext'])
        emitted.append((sp_, a_start, t_start))
    start = len(prog.ops)
    for sp_, a_start, t_start in emitted:
        prog.emit(Z_GENERATE, sp_['flags'],
                  (sp_['first'], sp_['count'], a_start, len(sp_['avoid']), t_start, sp_['meta_flags']),
                  (sp_['max_depth'],) + (tuple(float(v) for v in sp_['count_range']) if sp_['count_range'] else (0., 0.)))
    prog.sections['reset'] = (start, len(prog.ops) - start)
    prog.reset_template = state


def _check_outline_caps(prog):
    """Outlines with more than MOOG_MAX_VERTS vertices (up to MOOG_MAX_OUTLINE) can be moved
    and drawn, but the overlap / collision kernels spend one lane per vertex: a layer that holds
    such a sprite must not appear in any op that tests overlaps."""
    def layers_of_list(start, count):
        return [prog.ipool[start + k] for k in range(count)]

    geom = set()
    for o in prog.ops:
        k, i = o['kind'], o['i']
        if k in (F_COLLISION, R_VANISH_ON_CONTACT, SC_CONTACT_COUNT):
            geom.update(i[0:2])
        elif k in (R_MODIFY_ON_CONTACT, T_CONTACT_REWARD, SC_CONTACT_ANY_COUNT):
            geom.update(layers_of_list(i[0], i[1]) + layers_of_list(i[2], i[3]))
        elif k == R_CREATE_SPRITES and i[3] > 0:
            geom.update([i[0]] + layers_of_list(i[2], i[3]))
        elif k == Z_GENERATE:
            slots = [i[0]] + [prog.ipool[i[2] + q] for q in range(i[3])]
            for s in slots:
                geom.add(max(l for l in range(prog.n_layers) if prog.layer_off[l] <= s))
    for l in sorted(geom):
        if prog.layer_vcap[l] > MAX_VERTS:
            raise CompileError(
                'layer {!r} holds a sprite with {} vertices and takes part in overlap tests; '
                'only outlines of at most {} vertices can (larger ones, up to {}, can be moved and drawn)'.format(
                    prog.layer_names[l], prog.layer_vcap[l], MAX_VERTS, MAX_OUTLINE))


def _scalar_kind(v):
    """0 python number (weak), 1 float32, 2 float64 -- how NumPy will promote
    the value in `angle + dt * angle_vel` (sprite.py:426-430)."""
    dt = getattr(v, 'dtype', None)
    if dt is None:
        return 0
    return 1 if dt == np.float32 else 2


def _sprite_flags(sp):
    flags = SF_CIRCLE if sp.shape == 'circle' else 0
    if getattr(sp.velocity, 'dtype', None) == np.float32:
        flags |= SF_VEL32
    flags |= _scalar_kind(sp.angle_vel) << SF_ANGVEL_SHIFT
    flags |= _scalar_kind(sp.angle) << SF_ANG_SHIFT
    return flags


class ShapeTable(object):
    """Deduplicated table of COM-centred unit outlines."""

    def __init__(self):
        self._index = {}
        self.verts = []
        self.nv = []
        self.names = []     # Sprite.shape of the first sprite that showed the outline ('square', ..., 'custom')

    def add(self, outline, name=None):
        outline = np.ascontiguousarray(outline, dtype=np.float64)
        key = outline.tobytes()
        sid = self._index.get(key)
        if sid is None:
            n = len(outline)
            if n > MAX_OUTLINE:
                raise CompileError(
                    'sprite outline has {} vertices; the device path supports '
                    'at most {}'.format(n, MAX_OUTLINE))
            if n < 3:
                raise CompileError('sprite outline needs at least 3 vertices')
            sid = len(self.nv)
            padded = np.zeros((MAX_OUTLINE, 2))
            padded[:n] = outline
            self.verts.append(padded)
            self.nv.append(n)
            self.names.append(name if isinstance(name, str) else 'custom')
            self._index[key] = sid
        return sid

    def arrays(self):
        n = max(len(self.nv), 1)
        verts = np.zeros((n, MAX_OUTLINE, 2))
        nv = np.zeros(n, dtype=np.int32)
        if self.nv:
            verts[:len(self.nv)] = np.stack(self.verts)
            nv[:len(self.nv)] = self.nv
        return verts, nv


def pack_states(prog, states, shape_table=None):
    """States -> dict of numpy arrays laid out as the device state record.

    Reads each sprite through the attributes shared by the reference's Sprite
    (sprite.py:261-327) and this repo's: position, velocity, angle, angle_vel,
    mass, scale, aspect_ratio, color, opacity, shape, max_radius and the
    private `_shape_path.vertices` / `_x_y_rotational_inertia`.
    """
    fixed_table = getattr(prog, 'shape_table', None)
    if fixed_table is not None and shape_table is None:
        shape_table = fixed_table
    table = ShapeTable() if shape_table is None else shape_table
    n, S, L = len(states), prog.n_slots, prog.n_layers
    dyn = np.zeros((n, DYN_FIELDS, S))
    stat = np.zeros((n, STAT_FIELDS, S))
    stat[:, 0, :] = 1.0  # mass of unused slots: harmless, never read
    stat[:, 1, :] = 1.0
    stat[:, 2, :] = 1.0
    meta = np.zeros((n, META_FIELDS, S), dtype=np.int32)
    vtx = np.zeros((n, max(prog.n_vtx, 1), 2))
    cnt = np.zeros((n, MAX_LAYERS), dtype=np.int32)
    shared_per_env = []
    for e, st in enumerate(states):
        shared = {}
        shared_per_env.append(shared)
        for l, name in enumerate(prog.layer_names):
            sprites = st[name]
            if len(sprites) > prog.layer_cap[l]:
                raise CompileError(
                    'layer {!r} holds {} sprites, capacity is {}'.format(
                        name, len(sprites), prog.layer_cap[l]))
            cnt[e, l] = len(sprites)
            for k, sp in enumerate(sprites):
                s = prog.layer_off[l] + k
                pos, vel = sp.position, sp.velocity
                dyn[e, :, s] = (pos[0], pos[1], vel[0], vel[1],
                                float(sp.angle), float(sp.angle_vel))
                ixy = sp._x_y_rotational_inertia  # pylint: disable=protected-access
                col = sp.color
                stat[e, :, s] = (float(sp.mass), float(sp.scale),
                                 float(sp.aspect_ratio), ixy[0], ixy[1],
                                 float(sp.max_radius), float(col[0]),
                                 float(col[1]), float(col[2]),
                                 float(sp.opacity))
                base = sp._shape_path.vertices[:-1]  # pylint: disable=protected-access
                meta[e, 0, s] = table.add(base, getattr(sp, 'shape', None))
                if fixed_table is not None and table is fixed_table and meta[e, 0, s] >= prog.n_table_shapes:
                    raise CompileError(
                        'a sprite of layer {!r} has a shape no sample state showed at compile time; rules that '
                        'assign scale / aspect_ratio need every shape in the program\'s shape table'.format(name))
                meta[e, 1, s] = _sprite_flags(sp)
                world = np.asarray(sp.vertices, dtype=np.float64)
                if len(world) > prog.layer_vcap[l]:
                    raise CompileError(
                        'a sprite of layer {!r} has {} vertices, more than any '
                        'sample state showed ({})'.format(
                            name, len(world), prog.layer_vcap[l]))
                meta[e, 2, s] = len(world)
                vtx[e, prog.voff[s]:prog.voff[s] + len(world)] = world
                if isinstance(vel, np.ndarray):
                    shared.setdefault(id(vel), []).append(s)
    envi = np.zeros((n, ENVI_WORDS), dtype=np.int32)
    # Sprites that hold the SAME velocity ndarray object (`Tether(update_angle_vel=False)` hands one
    # array to every tethered sprite, tether_physics.py:86-91) share later in-place updates: they
    # get a common alias id (MOOG_SF_VALIAS_SHIFT), numbered in slot order
    for e in range(n):
        next_id = 0
        for slots in sorted(shared_per_env[e].values(), key=min):
            if len(slots) > 1:
                next_id += 1
                for s in slots:
                    meta[e, 1, s] |= next_id << SF_VALIAS_SHIFT
        envi[e, EI_VALIAS_NEXT] = next_id
    envf = np.zeros((n, max(prog.n_envf, 1)))
    if prog.maze_offsets:
        from . import host_maze
        for e, st in enumerate(states):
            for layer, off in prog.maze_offsets.items():
                envf[e, off:off + host_maze.MAZE_WORDS] = host_maze.maze_record(st[layer])
    if getattr(prog, 'meta_vars', None):     # the env's meta_state variables as meta_state_initializer() leaves them
        values = prog.meta_values()
        envf[:, prog.meta_var_off:prog.meta_var_off + len(values)] = values
    meta_keys = getattr(prog, 'meta_keys', None)
    if meta_keys:
        # sprite.metadata[key] for the keys the program's callables read; NaN where a sprite has no such
        # key (the reference would raise KeyError there) -- bools and numbers only
        S = prog.n_slots
        envf[:, prog.meta_off:prog.meta_off + len(meta_keys) * S] = np.nan
        for e, st in enumerate(states):
            for l, name in enumerate(prog.layer_names):
                for k, sp in enumerate(st[name]):
                    md = getattr(sp, 'metadata', None)
                    if not isinstance(md, dict):
                        continue
                    for c, key in enumerate(meta_keys):
                        if key in md:
                            v = md[key]
                            if v is None or not (isinstance(v, (bool, int, float)) or hasattr(v, '__float__')):
                                raise CompileError('sprite.metadata[{!r}] = {!r}: only numbers and bools are carried on '
                                                   'the device'.format(key, v))
                            envf[e, prog.meta_off + c * S + prog.layer_off[l] + k] = float(v)
    shape_verts, shape_nv = table.arrays()
    return dict(dyn=dyn, stat=stat, meta=meta, vtx=vtx, cnt=cnt, envi=envi,
                envf=envf, shape_verts=shape_verts, shape_nv=shape_nv,
                shape_table=table)


def unpack_state(prog, arrays, e):
    """Inverse of pack_states for env `e`: {layer: [dict of factors]}."""
    out = collections.OrderedDict()
    for l, name in enumerate(prog.layer_names):
        rows = []
        for k in range(int(arrays['cnt'][e, l])):
            s = prog.layer_off[l] + k
            d = arrays['dyn'][e, :, s]
            t = arrays['stat'][e, :, s]
            rows.append(dict(
                x=d[0], y=d[1], x_vel=d[2], y_vel=d[3], angle=d[4],
                angle_vel=d[5], mass=t[0], scale=t[1], aspect_ratio=t[2],
                c0=t[6], c1=t[7], c2=t[8], opacity=t[9],
                shape_id=int(arrays['meta'][e, 0, s])))
        out[name] = rows
    return out
