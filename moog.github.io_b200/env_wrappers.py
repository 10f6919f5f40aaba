"""Batched counterparts of the reference's env wrappers (moog/env_wrappers/).

`VectorGymWrapper` gives a `BatchedEnvironment` the (obs, reward, done, info)
protocol of the reference's `GymWrapper` (gym_wrapper.py:48-140), one entry per
env, without depending on `gym`: spaces are described by plain dicts.
`BatchedSimulation` is the snapshot / restore facility of
`SimulationEnvironment` (simulation.py:55-83) for tree search: the whole batch
is saved to and restored from device tensors.

Host-side convenience only; the step itself is `BatchedEnvironment.step`.
"""
import json
import os
import time
from datetime import datetime

import numpy as np
import torch

from . import compiler
from .batched_env import STEP_FIRST, STEP_LAST


class VectorGymWrapper(object):
    """Gym-style vector env over a BatchedEnvironment (auto-resetting)."""

    metadata = {'render.modes': ['rgb_array']}

    def __init__(self, env):
        self._env = env
        self._last_render = None
        self._env.reset()

    @property
    def num_envs(self):
        return self._env.num_envs

    @property
    def observation_space(self):
        """{key: dict(low, high, shape, dtype)} per env (gym_wrapper.py:66-78)."""
        spaces = {}
        for key, r in self._env.program.views:
            spaces[key] = dict(low=0, high=255, shape=(r['height'], r['width'], 3), dtype='uint8')
        for key, m in self._env.program.masks:  # SpriteMask: a record slot per pixel, -1 for none
            spaces[key] = dict(low=-1, high=self._env.program.n_slots - 1, shape=(m['height'], m['width']),
                               dtype='int16')
        for key, r in self._env.program.rays:  # RaySensor: (t / max_range, slot) per ray, (1, -1) for none
            spaces[key] = dict(low=-1, high=max(1, self._env.program.n_slots - 1), shape=(r['num_rays'], 2),
                               dtype='float32')
        key = self._env.program.state_key
        if key is not None:
            spaces[key] = dict(low=-np.inf, high=np.inf, shape=(self._env.program.n_slots, compiler.OBS_COLS),
                               dtype='float32')
        return spaces

    @property
    def action_space(self):
        """One entry per action-space component, in `program.action_layout` order:
        Joystick / SetPosition -> Box(-1, 1, (2,)) resp. Box(0, 1, (2,)), Grid -> Discrete(5)."""
        out = []
        for key, kind, _, width in self._env.program.action_layout:
            if kind == 'Grid':
                out.append(dict(key=key, type='Discrete', n=5))
            else:
                low = 0. if kind == 'SetPosition' else -1.
                out.append(dict(key=key, type='Box', low=low, high=1., shape=(width,), dtype='float32'))
        return out

    def _obs(self, ts):
        obs = dict(ts.observation)
        if 'image' in obs:
            self._last_render = obs['image']
        return obs

    def reset(self):
        return self._obs(self._env.reset())

    def step(self, action):
        """-> obs {key: tensor[N, ...]}, reward float32[N] (0 where dm_env has None),
        done bool[N], info {'discount': float32[N]}.  An env that is done is reset by
        the next call (environment.py:100-101), which ignores that env's action."""
        ts = self._env.step(action)
        reward = torch.nan_to_num(ts.reward, nan=0.0)
        done = ts.step_type == STEP_LAST
        return self._obs(ts), reward, done, {'discount': ts.discount}

    def render(self, mode='rgb_array'):
        del mode
        return self._last_render

    def close(self):
        pass


class BatchedSimulation(object):
    """Snapshot / restore of a whole batch (simulation.py:55-83): `SimulationEnvironment`'s
    protocol -- `reset`, `step`, `sim_step`, `sim_pop(index)` -- plus explicit `push` / `pop`.
    A snapshot is every array of the state record (task / action-space / rule memory lives in
    it: `envf`, `envi`) and the last TimeStep's scalars."""

    def __init__(self, env):
        self._env = env
        self._stack = []

    def _snapshot(self):
        e = self._env.engine
        return (self._env.state_dict(), e.reward.clone(), e.step_type.clone(), e.discount.clone())

    def _restore(self, snap):
        sd, reward, step_type, discount = snap
        self._env.load_state_dict(sd)
        e = self._env.engine
        e.reward.copy_(reward)
        e.step_type.copy_(step_type)
        e.discount.copy_(discount)

    def push(self):
        self._stack.append(self._snapshot())
        return len(self._stack)

    def pop(self):
        if not self._stack:
            raise IndexError('no snapshot to restore')
        self._restore(self._stack.pop())

    def reset(self):
        """simulation.py:60-62"""
        self._stack = []
        return self._env.reset()

    def step(self, action):
        """simulation.py:64-69: a real step first discards every simulated one."""
        if self._stack:
            self.sim_pop(index=0)
        self._stack = []
        return self._env.step(action)

    def sim_step(self, action):
        """simulation.py:71-87: snapshot, then step.  The reference refuses to simulate across an
        episode boundary (returns None when the env is about to reset); for a batch that is
        `None` as soon as ANY env is pending a reset."""
        if bool((self._env.engine.state.envi[:, 1] != 0).any()):    # MOOG_EI_RESET_NEXT
            return None
        self._stack.append(self._snapshot())
        return self._env.step(action)

    def sim_pop(self, index=-1):
        """simulation.py:89-100: restore snapshot `index`, drop it and everything after it."""
        self._restore(self._stack[index])
        self._stack = self._stack[:index]

    @property
    def stack_depth(self):
        return len(self._stack)


# ---------------------------------------------------------------------------
# logger.py: episode logs in the reference's wire format
# ---------------------------------------------------------------------------
_FILENAME_ZFILL = 5          # logger.py:27
FACTOR_NAMES = ('x', 'y', 'shape', 'angle', 'scale', 'aspect_ratio', 'c0', 'c1', 'c2', 'opacity',
                'x_vel', 'y_vel', 'angle_vel', 'mass', 'metadata')      # sprite.py:237-241


class VertexLogging(object):
    NEVER = 'NEVER'
    ALWAYS = 'ALWAYS'
    WHEN_NECESSARY = 'WHEN_NECESSARY'


class BatchedLoggingEnvironment(object):
    """`LoggingEnvironment` (moog/env_wrappers/logger.py:73-224) for chosen envs of a batch.

    Every logged env gets a directory `<log_dir>/<timestamp>/env_<n>/` laid out exactly like the
    reference's log directory: `attributes.txt` (the JSON list of logged attributes: the 15 sprite
    factors + `id`), `description.txt`, and one file per episode, `00000`, `00001`, ..., holding the
    JSON list of that episode's steps,

        [['time', t], ['reward', r], ['step_type', v], ['action', a], ['meta_state', None], state]
        state = [[layer_name, [sprite_attributes, ...]], ...]

    with `reward` None on a FIRST step, `step_type` the dm_env.StepType value and the vertices
    appended to a sprite's attribute list according to `log_vertices` (logger.py:186-195), so
    moog_demos/restore_logged_data.py reads these logs unchanged.  What the device does not carry is
    logged as: `metadata` None, `meta_state` None; `id` is `1000 * episode + slot` of the sprite --
    a sprite keeps its id while its layer keeps its length, and when a layer changes length
    (VanishOnContact ...) the sprites of that layer are treated as new (WHEN_NECESSARY logs their
    vertices again), so that vertices can always be resolved by id as the reference promises.
    The rows of the logged envs are read back from the device every step: a debugging / data
    collection tool, not a fast path (logger.py:6-13 says the same of the reference).
    """

    def __init__(self, env, log_dir='logs', log_vertices='WHEN_NECESSARY', envs=(0,)):
        if not hasattr(VertexLogging, log_vertices):
            raise ValueError('log_vertices is {} but must be in VertexLogging values'.format(log_vertices))
        self._env = env
        self._log_vertices = log_vertices
        self._envs = [int(n) for n in envs]
        now_str = datetime.now().strftime('%Y_%m_%d_%H_%M_%S')
        root = os.path.join(log_dir if log_dir[0] == '/' else os.path.join(os.getcwd(), log_dir), now_str)
        self._attributes = list(FACTOR_NAMES) + ['id']
        self._dirs = {}
        for n in self._envs:
            d = os.path.join(root, 'env_{}'.format(n))
            os.makedirs(d)
            self._dirs[n] = d
            with open(os.path.join(d, 'attributes.txt'), 'w') as f:
                json.dump(self._attributes, f)
            with open(os.path.join(d, 'description.txt'), 'w') as f:
                f.write(self._description())
        self.log_dir = root
        self._episode_count = {n: 0 for n in self._envs}
        self._episode_log = {n: [] for n in self._envs}
        self._known = {n: {} for n in self._envs}      # layer -> count when its vertices were last logged
        self._idx = torch.as_tensor(self._envs, device=env.engine.device, dtype=torch.long)

    def _description(self):
        text = ('Each numerical file in this directory is an episode of the task. Each such file contains a '
                'json-serialized list, each element of which represents an environment step in the episode. Each step '
                'is a list of four elements, [[`time`, time], [`reward`, reward], [`step_type`, step_type], [`action`, '
                'action], [`meta_state`, meta_state`], state].\n\n\n\ntime is a timestamp of the timestep.\n\n\n\n'
                'reward contains the value of the reward at that step.\n\n\n\nstep_type indicates the '
                'dm_env.StepType of that step, i.e. whether it was first, mid, or last.\n\n\n\naction contains the '
                'agent action for the step.\n\n\n\nmeta_state is the serialized meta_state of the environment.'
                '\n\n\n\nstate is a list, each element of which represents a layer in the environment state. The layer '
                'is represented as a list [k, [], [], [], ...], where k is the layer name and the subsequent elements are '
                'serialized sprites. Each serialized sprite is a list of attributes. See attributes.txt for the '
                'attributes contained.')
        if self._log_vertices == VertexLogging.ALWAYS:
            text += ' Furthermore, a list of vertices is appended to the attribute list for each serialized sprite.'
        elif self._log_vertices == VertexLogging.WHEN_NECESSARY:
            text += ('\n\n\n\nFurthermore, a list of vertices is appended to the attribute list for a serialized for '
                     'the first timestep in which that serialized sprite appears, or when the sprite has changed shape.')
        return text

    # -- protocol ---------------------------------------------------------------
    def reset(self):
        ts = self._env.reset()
        for n in self._envs:
            self._known[n] = {}
        return ts

    def step(self, action=None):
        ts = self._env.step(action)
        self._log(ts, action)
        return ts

    def __getattr__(self, name):
        return getattr(self._env, name)

    def _unflatten_action(self, row):
        """One env's action as the reference's caller passed it (logger.py:203 serialises that): a Grid
        index as an int, a Joystick / SetPosition action as two floats, a Composite as a dict of those."""
        parts = {}
        for key, kind, off, width in self._env.program.action_layout:
            parts[key] = int(row[off]) if kind == 'Grid' else [float(v) for v in row[off:off + width]]
        if list(parts.keys()) == [None]:
            return parts[None]
        return parts

    # -- serialisation ------------------------------------------------------------
    def _log(self, ts, action):
        env, prog = self._env, self._env.program
        st = env.engine.state
        rows = {k: getattr(st, k).index_select(0, self._idx).cpu().numpy() for k in ('dyn', 'stat', 'meta', 'cnt', 'vtx', 'envi')}
        step_type = ts.step_type.index_select(0, self._idx).cpu().numpy()
        reward = ts.reward.index_select(0, self._idx).cpu().numpy()
        act = None
        if action is not None:
            a = env._flatten_action(action)  # pylint: disable=protected-access
            a = a if torch.is_tensor(a) else torch.as_tensor(np.asarray(a))
            act = a.reshape(env.num_envs, -1)[self._idx.to(a.device)].cpu().numpy()
        names = self._env.shape_names()
        now = time.time()
        for k, n in enumerate(self._envs):
            first = int(step_type[k]) == STEP_FIRST
            if first:
                self._known[n] = {}
            state = []
            episode = int(rows['envi'][k][3])
            for l, layer in enumerate(prog.layer_names):
                count = int(rows['cnt'][k][l])
                fresh = self._known[n].get(layer) != count
                self._known[n][layer] = count
                sprites = []
                for j in range(count):
                    s = prog.layer_off[l] + j
                    d, t, m = rows['dyn'][k][:, s], rows['stat'][k][:, s], rows['meta'][k][:, s]
                    sid = int(m[0])
                    attrs = [float(d[0]), float(d[1]), names[sid] if sid < len(names) else 'custom', float(d[4]),
                             float(t[1]), float(t[2]), float(t[6]), float(t[7]), float(t[8]), float(t[9]),
                             float(d[2]), float(d[3]), float(d[5]), float(t[0]), None, 1000 * episode + s]
                    if self._log_vertices == VertexLogging.ALWAYS or (
                            self._log_vertices == VertexLogging.WHEN_NECESSARY and fresh):
                        v0 = prog.voff[s]
                        attrs.append(rows['vtx'][k][v0:v0 + int(m[2])].tolist())
                    sprites.append(attrs)
                state.append([layer, sprites])
            r = None if (first or np.isnan(reward[k])) else float(reward[k])
            # dm_env.StepType: FIRST 0, MID 1, LAST 2
            step = [['time', now], ['reward', r], ['step_type', int(step_type[k])],
                    ['action', None if act is None else self._unflatten_action(act[k])],
                    ['meta_state', self._env.meta_state(int(n))], state]
            self._episode_log[n].append(step)
            if int(step_type[k]) == STEP_LAST:
                fn = os.path.join(self._dirs[n], str(self._episode_count[n]).zfill(_FILENAME_ZFILL))
                with open(fn, 'w') as f:
                    json.dump(self._episode_log[n], f)
                self._episode_count[n] += 1
                self._episode_log[n] = []
