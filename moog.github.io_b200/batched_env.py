"""BatchedEnvironment: N independent MOOG environments stepped on one B200.

Mirrors `moog.environment.Environment` (reference moog/environment.py:28-131):
same constructor arguments -- so `BatchedEnvironment(**get_config(level),
num_envs=N)` works on an unchanged MOOG config -- and the same `reset()` /
`step(action)` / `observation()` protocol, with every TimeStep field batched:

    step_type   int32  [N]   0 FIRST, 1 MID, 2 LAST        (dm_env.StepType)
    reward      float32[N]   NaN on FIRST steps            (dm_env: None)
    discount    float32[N]   1 mid, 0 last, NaN first
    observation {'image': uint8 [N, H, W, 3]}              (PILRenderer; each one of the config's
                                                           PILRenderers under its own key)
                {key: float32 [N, S, 16]}                 (RawState: every sprite slot, see
                                                           include/moog_b200_program.h MOOG_OBS_*)
                {key: int16 [N, H, W]}                    (SpriteMask: the slot each pixel shows,
                                                           -1 for none)
                {key: float32 [N, R, 2]}                  (RaySensor: t / max_range and the slot
                                                           each ray meets first, (1, -1) for none)

An env whose previous step returned LAST is reset by the next `step()` call and
ignores that call's action (environment.py:100-101).  Initial states come from
a pool produced by the config's own `state_initializer` on the host and kept
on the device; which pool entry a resetting env receives is drawn on the device.

PyTorch is used for device memory and streams only.  All arithmetic happens in
libmoog_b200.so (include/moog_b200.h); there is no fallback path.
"""
import collections
import contextlib
import ctypes
import time

import numpy as np
import torch

from . import capi
from . import compiler

TimeStep = collections.namedtuple(
    'TimeStep', ['step_type', 'reward', 'discount', 'observation'])

STEP_FIRST, STEP_MID, STEP_LAST = 0, 1, 2

_ERR_TEXT = {
    1: 'ValueError: collision normal is not a unit vector (collisions.py:323-326)',
    2: 'RuntimeError: _position_correction would not terminate (collisions.py:740)',
    4: 'ValueError: TetherZippedLayers layers differ in length (tether_physics.py:192-196)',
    8: 'RuntimeError: layer capacity exceeded',
    16: 'ValueError: Object is not on the maze grid (maze_physics.py:93-104)',
    32: 'RecursionError: max_recursion_depth exceeded trying to initialize a non-overlapping sprite '
        '(sprite_generators.py:92-98) / ValueError: maximum number of tries exceeded (distributions.py:341-349)',
    64: 'ValueError: There must be an even number of portals (portal.py:49-52)',
    128: 'IndexError: a condition / reward function indexed state[layer][i] beyond the sprites the layer holds',
}

_STATE_DTYPES = dict(dyn=torch.float64, stat=torch.float64, meta=torch.int32,
                     cnt=torch.int32, envi=torch.int32, envf=torch.float64,
                     vtx=torch.float64)


class DeviceState(object):
    """The SoA state record of n envs as torch tensors on one device."""

    KEYS = ('dyn', 'stat', 'meta', 'cnt', 'envi', 'envf', 'vtx')

    def __init__(self, program, n, device):
        S, VT = program.n_slots, max(program.n_vtx, 1)
        self.n = n
        self.device = torch.device(device)
        z = lambda shape, k: torch.zeros(shape, dtype=_STATE_DTYPES[k], device=self.device)
        self.dyn = z((n, compiler.DYN_FIELDS, S), 'dyn')
        self.stat = z((n, compiler.STAT_FIELDS, S), 'stat')
        self.meta = z((n, compiler.META_FIELDS, S), 'meta')
        self.cnt = z((n, compiler.MAX_LAYERS), 'cnt')
        self.envi = z((n, compiler.ENVI_WORDS), 'envi')
        self.envf = z((n, max(program.n_envf, 1)), 'envf')
        self.vtx = z((n, VT, 2), 'vtx')

    def upload(self, arrays, rows=None):
        """arrays: dict from compiler.pack_states (numpy); rows: env indices."""
        for k in self.KEYS:
            src = torch.from_numpy(np.ascontiguousarray(arrays[k])).to(
                self.device, dtype=_STATE_DTYPES[k])
            dst = getattr(self, k)
            if rows is None:
                if src.shape != dst.shape:
                    raise ValueError('{}: shape {} != {}'.format(k, tuple(src.shape), tuple(dst.shape)))
                dst.copy_(src)
            else:
                dst[rows] = src

    def download(self):
        return {k: getattr(self, k).cpu().numpy() for k in self.KEYS}

    def clone(self):
        out = object.__new__(DeviceState)
        out.n, out.device = self.n, self.device
        for k in self.KEYS:
            setattr(out, k, getattr(self, k).clone())
        return out

    def copy_from(self, other):
        for k in self.KEYS:
            getattr(self, k).copy_(getattr(other, k))

    def struct(self, first=0):
        """`moog_state` of the envs [first, n): the row pointers of env `first`."""
        if first == 0:
            # the tensors are allocated once and only ever written in place
            key = tuple(getattr(self, k).data_ptr() for k in self.KEYS)
            cached = getattr(self, '_struct0', None)
            if cached is None or cached[0] != key:
                cached = (key, capi.MoogState(*key))
                self._struct0 = cached
            return cached[1]
        ptrs = []
        for k in self.KEYS:
            t = getattr(self, k)
            ptrs.append(t.data_ptr() + first * t.stride(0) * t.element_size())
        return capi.MoogState(*ptrs)

    def nbytes(self):
        return sum(getattr(self, k).numel() * getattr(self, k).element_size() for k in self.KEYS)


_NULL_CONTEXT = contextlib.nullcontext()


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


class Engine(object):
    """Program + state + the raw C-ABI calls (used by BatchedEnvironment and
    directly by the parity tests / bench)."""

    def __init__(self, program, num_envs, device='cuda', seed=0):
        if not torch.cuda.is_available():
            raise capi.MoogError('moog_b200 needs a CUDA device; there is no CPU path')
        self.program = program
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise capi.MoogError('device must be a CUDA device')
        self.n = int(num_envs)
        self.seed = int(seed)
        self._check_views(program)
        with torch.cuda.device(self.device):
            self.dev_program = capi.DeviceProgram(program.blob)
        self.dev_program.set_option('seed', self.seed & 0x7fffffff)
        self.state = DeviceState(program, self.n, self.device)
        self.pool = None
        f32 = dict(dtype=torch.float32, device=self.device)
        self.reward = torch.zeros(self.n, **f32)
        self.discount = torch.zeros(self.n, **f32)
        self.step_type = torch.zeros(self.n, dtype=torch.int32, device=self.device)
        self.counters = torch.zeros((self.n, 8), dtype=torch.int64, device=self.device)
        self.stats = torch.zeros(4, dtype=torch.float64, device=self.device)
        # view 0 (the first PILRenderer) in `frames`, the further ones in `view_frames`, in view order
        views = [r for _, r in getattr(program, 'views', ())] or (
            [program.render] if program.render is not None else [])
        frames = [torch.zeros((self.n, r['height'], r['width'], 3), dtype=torch.uint8, device=self.device)
                  for r in views]
        self.frames = frames[0] if frames else None
        self.view_frames = frames[1:]
        # one int16 [N, H, W] buffer per SpriteMask, in mask order
        self.masks = [torch.full((self.n, m['height'], m['width']), -1, dtype=torch.int16, device=self.device)
                      for _, m in getattr(program, 'masks', ())]
        # one float32 [N, R, 2] buffer per RaySensor, in sensor order, and the moog_ray_spec of each, whose
        # direction table is uploaded once here
        self.rays = []
        self._ray_specs = []
        for _, r in getattr(program, 'rays', ()):
            self.rays.append(torch.empty((self.n, r['num_rays'], 2), **f32))
            dirs = torch.from_numpy(r['dirs']).to(self.device, dtype=torch.float64).contiguous()
            spec = capi.MoogRaySpec(r['agent_layer'], r['agent_index'], r['layers'], r['num_rays'],
                                    r['max_range'], dirs.data_ptr())
            self._ray_specs.append((spec, dirs))
        self.sprites = None
        if getattr(program, 'state_key', None) is not None:
            self.sprites = torch.zeros((self.n, program.n_slots, compiler.OBS_COLS), **f32)
        self._calls = 0
        self._pinned_ok = set()

    # -- helpers -----------------------------------------------------------
    @staticmethod
    def _check_views(program):
        """Every renderer must be drawable by the render kernel (moog_render_plan): a view that no
        chunk of its canvas fits one CTA's shared memory is refused here, before anything is
        allocated or launched."""
        views = list(getattr(program, 'views', ())) or (
            [('image', program.render)] if program.render is not None else [])
        for v, (key, r) in enumerate(views):
            code, _, _ = capi.render_plan(program.blob, v)
            if code == capi.E_UNSUPPORTED:
                raise capi.MoogError(
                    'observer {!r}: PILRenderer(image_size=({}, {}), anti_aliasing={}) draws a {} x {} canvas, '
                    'and no chunk of it fits the shared memory of one CTA'.format(
                        key, r['width'], r['height'], r['aa'], r['aa'] * r['width'], r['aa'] * r['height']))
            capi.check(code)
        for k, (key, m) in enumerate(getattr(program, 'masks', ())):
            code, _, _ = capi.mask_plan(program.blob, k)
            if code == capi.E_UNSUPPORTED:
                raise capi.MoogError(
                    'observer {!r}: SpriteMask(image_size=({}, {})) cannot be drawn: no band of its rows fits '
                    'the shared memory of one CTA next to the edge lists of its sprites'.format(
                        key, m['width'], m['height']))
            capi.check(code)

    def call_seed(self):
        """io.seed of the next env_step call (a different Philox key every call)."""
        return (self.seed * 0x9E3779B97F4A7C15 + self._calls) & 0xFFFFFFFFFFFFFFFF

    def _on_device(self):
        """Context that makes this engine's GPU current (free when it already is)."""
        index = self.device.index
        if index is None or torch.cuda.current_device() == index:
            return _NULL_CONTEXT
        return torch.cuda.device(self.device)

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check_reachable(self, out, what):
        """`out` is on this device or in pinned host memory (the kernels store into it)."""
        if out.device.type == 'cpu':
            if out.data_ptr() not in self._pinned_ok:
                if not out.is_pinned():
                    raise ValueError('host {} must live in pinned memory'.format(what))
                self._pinned_ok.add(out.data_ptr())
        elif out.device != self.state.dyn.device:
            raise ValueError('{} are on {}, the envs on {}'.format(what, out.device, self.state.dyn.device))

    def set_pool(self, arrays):
        n = arrays['dyn'].shape[0]
        self.pool = DeviceState(self.program, n, self.device)
        self.pool.upload(arrays)

    def _as_f64(self, x, width):
        if x is None:
            return None
        if not torch.is_tensor(x):
            x = torch.as_tensor(np.asarray(x))
        x = x.to(self.device, dtype=torch.float64, non_blocking=True).reshape(self.n, -1)
        if x.shape[1] != width:
            raise ValueError('expected [{}, {}], got {}'.format(self.n, width, tuple(x.shape)))
        return x.contiguous()

    # -- C-ABI calls ---------------------------------------------------------
    def post_reset(self, rule_noise=None):
        rn = self._as_f64(rule_noise, self.program.rule_noise_dim) if rule_noise is not None else None
        st = self.state.struct()
        with torch.cuda.device(self.device):
            capi.check(capi.lib().moog_env_post_reset(
                self.dev_program.handle, ctypes.byref(st), self.n, _ptr(rn), self._stream()))

    def env_step(self, actions=None, noise=None, rule_noise=None, auto_reset=True,
                 reset_index=None, want_counters=False, sample_resets=False, frames=None):
        """`moog_env_step`.  frames: None, True (draw the frame of the state every env is left in
        into `self.frames`) or a uint8 [N, H, W, 3] tensor to draw into -- on this device, or a
        pinned CPU tensor, which the kernels then write over PCIe as the envs finish."""
        p = self.program
        if frames is True:
            frames = self.frames
        if frames is not None:
            if self.frames is None:
                raise capi.MoogError('the program has no PILRenderer observer')
            if (frames.dtype != torch.uint8 or tuple(frames.shape) != tuple(self.frames.shape)
                    or not frames.is_contiguous()):
                raise ValueError('frames must be a contiguous uint8 tensor of shape {}'.format(
                    tuple(self.frames.shape)))
            self._check_reachable(frames, 'frames')
        act = self._as_f64(actions, max(p.action_dim, 1)) if actions is not None else None
        nz = self._as_f64(noise, p.K * p.noise_dim) if (noise is not None and p.noise_dim) else None
        rn = self._as_f64(rule_noise, p.rule_noise_dim) if (
            rule_noise is not None and p.rule_noise_dim) else None
        ri = None
        if reset_index is not None:
            ri = torch.as_tensor(reset_index).to(self.device, dtype=torch.int32).contiguous()
        io = capi.MoogStepIO()
        io.actions, io.noise, io.rule_noise = _ptr(act), _ptr(nz), _ptr(rn)
        pool_struct = None
        if auto_reset and self.pool is not None:
            pool_struct = self.pool.struct()
            io.pool = ctypes.pointer(pool_struct)
            io.pool_size = self.pool.n
        io.reset_index = _ptr(ri)
        io.sample_resets = 1 if sample_resets else 0
        io.seed = self.call_seed()
        io.reward, io.step_type, io.discount = _ptr(self.reward), _ptr(self.step_type), _ptr(self.discount)
        io.counters = _ptr(self.counters) if want_counters else None
        io.stats = _ptr(self.stats)
        io.frames = _ptr(frames)
        st = self.state.struct()
        with self._on_device():
            capi.check(capi.lib().moog_env_step(
                self.dev_program.handle, ctypes.byref(st), self.n, ctypes.byref(io), self._stream()))
        self._calls += 1

    def physics_step(self, noise=None, want_counters=True):
        p = self.program
        nz = self._as_f64(noise, p.K * p.noise_dim) if (noise is not None and p.noise_dim) else None
        st = self.state.struct()
        with torch.cuda.device(self.device):
            capi.check(capi.lib().moog_physics_step(
                self.dev_program.handle, ctypes.byref(st), self.n, _ptr(nz),
                _ptr(self.counters) if want_counters else None, self._stream()))

    def overlap_pairs(self, layer_a, layer_b):
        p = self.program
        la, lb = p.layer_index(layer_a), p.layer_index(layer_b)
        out = torch.zeros((self.n, p.layer_cap[la], p.layer_cap[lb]), dtype=torch.uint8, device=self.device)
        st = self.state.struct()
        with torch.cuda.device(self.device):
            capi.check(capi.lib().moog_overlap_pairs(
                self.dev_program.handle, ctypes.byref(st), self.n, la, lb, _ptr(out), self._stream()))
        return out

    @property
    def n_views(self):
        """PILRenderer observers of the program (0 without one)."""
        return 0 if self.frames is None else 1 + len(self.view_frames)

    def view_buffer(self, view):
        """This engine's frames of view `view`: `frames` for view 0, else `view_frames[view - 1]`."""
        if not 0 <= view < self.n_views:
            raise ValueError('view {} is outside [0, {})'.format(view, self.n_views))
        return self.frames if view == 0 else self.view_frames[view - 1]

    def render(self, out=None, first=0, count=None, view=0):
        """Frames of view `view` of the envs [first, first + count) into out[first:first + count]
        (`out` None: the view's own buffer).  A view other than 0 is drawn by `moog_render_view`
        into a contiguous uint8 [N, H, W, 3] tensor on this device or in pinned host memory, whose
        range starts 16-byte aligned."""
        if self.frames is None:
            raise capi.MoogError('the program has no PILRenderer observer')
        own = self.view_buffer(view)
        out = own if out is None else out
        count = self.n - first if count is None else count
        if first < 0 or count < 0 or first + count > self.n:
            raise ValueError('env range [{}, {}) is outside [0, {})'.format(first, first + count, self.n))
        if view != 0:
            if out.dtype != torch.uint8 or tuple(out.shape) != tuple(own.shape) or not out.is_contiguous():
                raise ValueError('frames of view {} must be a contiguous uint8 tensor of shape {}'.format(
                    view, tuple(own.shape)))
            self._check_reachable(out, 'frames')
        st = self.state.struct(first)
        dst = ctypes.c_void_p(out.data_ptr() + first * out.stride(0) * out.element_size())
        with torch.cuda.device(self.device):
            if view == 0:
                capi.check(capi.lib().moog_render(
                    self.dev_program.handle, ctypes.byref(st), count, dst, self._stream()))
            else:
                capi.check(capi.lib().moog_render_view(
                    self.dev_program.handle, ctypes.byref(st), count, view, dst, self._stream()))
        return out

    def render_mask(self, out=None, first=0, count=None, mask=0):
        """SpriteMask `mask` of the envs [first, first + count) into out[first:first + count] (`out` None:
        the mask's own buffer in `masks`), drawn by `moog_render_mask`: a contiguous int16 [N, H, W]
        tensor on this device or in pinned host memory, whose range starts 16-byte aligned."""
        if not 0 <= mask < len(self.masks):
            raise ValueError('mask {} is outside [0, {})'.format(mask, len(self.masks)))
        own = self.masks[mask]
        out = own if out is None else out
        count = self.n - first if count is None else count
        if first < 0 or count < 0 or first + count > self.n:
            raise ValueError('env range [{}, {}) is outside [0, {})'.format(first, first + count, self.n))
        if out.dtype != torch.int16 or tuple(out.shape) != tuple(own.shape) or not out.is_contiguous():
            raise ValueError('mask {} must be a contiguous int16 tensor of shape {}'.format(mask, tuple(own.shape)))
        self._check_reachable(out, 'masks')
        st = self.state.struct(first)
        dst = ctypes.c_void_p(out.data_ptr() + first * out.stride(0) * out.element_size())
        with self._on_device():
            capi.check(capi.lib().moog_render_mask(
                self.dev_program.handle, ctypes.byref(st), count, mask, dst, self._stream()))
        return out

    def sense_rays(self, out=None, first=0, count=None, sensor=0):
        """RaySensor `sensor` of the envs [first, first + count) into out[first:first + count] (`out` None:
        the sensor's own buffer in `rays`), cast by `moog_ray_sensor`: a contiguous float32 [N, R, 2]
        tensor on this device or in pinned host memory, whose range starts 16-byte aligned."""
        if not 0 <= sensor < len(self.rays):
            raise ValueError('sensor {} is outside [0, {})'.format(sensor, len(self.rays)))
        own = self.rays[sensor]
        out = own if out is None else out
        count = self.n - first if count is None else count
        if first < 0 or count < 0 or first + count > self.n:
            raise ValueError('env range [{}, {}) is outside [0, {})'.format(first, first + count, self.n))
        if out.dtype != torch.float32 or tuple(out.shape) != tuple(own.shape) or not out.is_contiguous():
            raise ValueError('rays of sensor {} must be a contiguous float32 tensor of shape {}'.format(
                sensor, tuple(own.shape)))
        self._check_reachable(out, 'rays')
        st = self.state.struct(first)
        dst = ctypes.c_void_p(out.data_ptr() + first * out.stride(0) * out.element_size())
        with self._on_device():
            capi.check(capi.lib().moog_ray_sensor(
                self.dev_program.handle, ctypes.byref(st), count, ctypes.byref(self._ray_specs[sensor][0]), dst,
                self._stream()))
        return out

    def observe_sprites(self, out=None):
        """`moog_observe_sprites`: RawState (raw_state.py:17-19) of every env as float32 [N, S, 16]
        (columns: include/moog_b200_program.h MOOG_OBS_*), into `self.sprites` or `out` -- a
        contiguous tensor of that shape on this device, or in pinned host memory, which the kernel
        then writes over PCIe.  Enqueued on the current stream behind whatever was enqueued before."""
        if out is None:
            if self.sprites is None:
                raise capi.MoogError('the program has no RawState observer')
            out = self.sprites
        shape = (self.n, self.program.n_slots, compiler.OBS_COLS)
        if out.dtype != torch.float32 or tuple(out.shape) != shape or not out.is_contiguous():
            raise ValueError('sprites must be a contiguous float32 tensor of shape {}'.format(shape))
        self._check_reachable(out, 'sprites')
        st = self.state.struct()
        with self._on_device():
            capi.check(capi.lib().moog_observe_sprites(
                self.dev_program.handle, ctypes.byref(st), self.n, _ptr(out), self._stream()))
        return out


class BatchedEnvironment(object):
    """See module docstring.  Reference: moog/environment.py:28-131."""

    def __init__(self, state_initializer, physics, task, action_space, observers,
                 game_rules=(), meta_state_initializer=None, *, num_envs,
                 device='cuda', pool_size=None, seed=0, layer_capacity=None,
                 initial_states=None, reset_mode='pool'):
        # (meta_state: None, or a dict of numbers / strings whose entries become variables of the env's
        # record -- compile_config refuses anything else)
        self.state_initializer = state_initializer
        self.num_envs = int(num_envs)
        config = dict(state_initializer=state_initializer, physics=physics, task=task,
                      action_space=action_space, observers=observers, game_rules=game_rules,
                      meta_state_initializer=meta_state_initializer)
        if initial_states is None:
            pool_size = int(pool_size or min(self.num_envs, 256))
            initial_states = [state_initializer() for _ in range(pool_size)]
        if reset_mode not in ('pool', 'device'):
            raise ValueError("reset_mode must be 'pool' or 'device'")
        self.reset_mode = reset_mode
        self.program = compiler.compile_config(config, initial_states, layer_capacity,
                                               reset_sampler=(reset_mode == 'device'))
        if reset_mode == 'device':
            # pool entry 0 is the template the device sampler starts every reset from
            initial_states = [self.program.reset_template] + list(initial_states)
        self._pool_arrays = compiler.pack_states(self.program, initial_states)
        self.engine = Engine(self.program, self.num_envs, device, seed)
        self.engine.set_pool(self._pool_arrays)
        self.action_space = action_space
        self.observers = observers
        # observers keys of the PILRenderers in view order (view 0 first)
        self._image_keys = [k for k, _ in self.program.views]
        self._image_key = self._image_keys[0] if self._image_keys else None
        self._state_key = self.program.state_key
        self._mask_keys = [k for k, _ in self.program.masks]   # SpriteMask observers in mask order
        self._ray_keys = [k for k, _ in self.program.rays]     # RaySensor observers in sensor order
        self._rng = np.random.RandomState(seed)
        self._started = False
        self._copy_stream = None
        self._copy_events = None
        self._auto_choice = None
        self._auto_calls = 0
        self._auto_times = {'mapped': [], 'chunked': []}

    # -- dm_env-like protocol -------------------------------------------------
    def _clear_envi(self):
        """Counters and error words back to 0 -- but not the two draw serials (MOOG_EI_CREATED,
        MOOG_EI_RULE_PASSES): they key the Philox draws of CreateSprites / random conditions, and an
        env reset by hand must not see the draws of its first episode again."""
        envi = self.engine.state.envi
        envi[:, :4].zero_()
        envi[:, 6:].zero_()

    def reset(self):
        """environment.py:82-96 for every env."""
        e = self.engine
        if self.reset_mode == 'device':
            # every env is marked terminated; the step kernel then resets it (environment.py:100-101)
            # and draws its generated sprites on the device
            for k in DeviceState.KEYS:
                getattr(e.state, k).copy_(getattr(e.pool, k)[0:1].expand_as(getattr(e.state, k)))
            self._clear_envi()
            e.state.envi[:, 1] = 1
            e.env_step(None, sample_resets=True)
            self._started = True
            return self._timestep()
        idx = torch.from_numpy(self._rng.randint(0, e.pool.n, size=self.num_envs)).to(e.device)
        for k in DeviceState.KEYS:
            if k == 'envi':
                self._clear_envi()
            else:
                getattr(e.state, k).copy_(getattr(e.pool, k).index_select(0, idx))
        e.post_reset()
        e.step_type.fill_(STEP_FIRST)
        e.reward.fill_(float('nan'))
        e.discount.fill_(float('nan'))
        self._started = True
        return self._timestep()

    def step(self, action=None):
        """environment.py:98-126 for every env; `action` is [N, action_dim]
        (Joystick: 2 floats, Grid: 1 index; Composite: dict of those or the
        concatenation in the order of `program.action_layout`)."""
        if not self._started:
            return self.reset()
        # the observation is drawn by the step call itself (inside the step kernel when a canvas
        # fits next to the env record, see include/moog_b200.h `frames`)
        self.engine.env_step(self._flatten_action(action), sample_resets=(self.reset_mode == 'device'),
                             frames=True if self._image_key is not None else None)
        return self._timestep(rendered=True)

    def shape_names(self):
        """Shape name of every shape id (meta row 0, column 2 of the RawState observation); an id beyond
        the list is a shape without a name."""
        table = self._pool_arrays.get('shape_table')
        return list(getattr(table, 'names', [])) if table is not None else []

    def step_to_host(self, action, host, chunks=4, frames='auto'):
        """`step(action)` whose TimeStep lands in the caller's pinned host buffers:
        `host` is a TimeStep of CPU tensors (step_type int32[N], reward float32[N],
        discount float32[N] or None, observation {'image': uint8[N,H,W,3]} -- one such image per
        PILRenderer, under its key -- and, with a RawState observer, its key -> pinned
        float32[N,S,16], with SpriteMask observers, each key -> pinned int16[N,H,W], and with RaySensor
        observers, each key -> pinned float32[N,R,2]).  Returns `host` once everything has arrived (the
        caller owns the TimeStep).  The other views, the masks, the rays and the sprite observation travel
        like the frames of view 0:
        stored by their kernels straight into the pinned tensors with 'mapped', computed in device
        memory and copied after it otherwise (with 'chunked': range by range, a view, mask or sensor whose
        per-env bytes are not a multiple of 16 in one range).

        frames = 'mapped': the step call draws every env's frame straight into the pinned host
        image (the kernels' stores cross PCIe while other envs are still being stepped; no
        device copy of the frames exists).  'device': the step call draws into device memory,
        one device-to-host copy follows.  'chunked': the step, then the frames rendered in
        `chunks` env ranges, the device-to-host copy of one range running on a second stream
        while the next range is rendered.  'auto': with a pinned host image the first 8 calls
        alternate between 'mapped' and 'chunked', time themselves, and the faster one is kept
        (mapped stores hide behind the step but move fewer bytes per second than the copy
        engines); 'device' when the image is not pinned."""
        img = host.observation[self._image_key] if self._image_key is not None else None
        more = [host.observation[k] for k in self._image_keys[1:]]  # views 1..
        spr = host.observation.get(self._state_key) if self._state_key is not None else None
        masks = [host.observation[k] for k in self._mask_keys]
        rays = [host.observation[k] for k in self._ray_keys]
        auto = frames == 'auto'
        if auto:
            frames = self._auto_frames(img)
        t_begin = time.perf_counter() if auto else 0.0
        if frames not in ('mapped', 'device', 'chunked'):
            raise ValueError("frames must be 'auto', 'mapped', 'device' or 'chunked'")
        e = self.engine
        main = torch.cuda.current_stream(e.device)
        if frames != 'chunked' or not self._started:
            if not self._started:
                self.reset()
                if img is not None:
                    img.copy_(e.frames, non_blocking=True)
                for dst, src in zip(more, e.view_frames):
                    dst.copy_(src, non_blocking=True)
                if spr is not None:
                    spr.copy_(e.sprites, non_blocking=True)
                for dst, src in zip(masks, e.masks):
                    dst.copy_(src, non_blocking=True)
                for dst, src in zip(rays, e.rays):
                    dst.copy_(src, non_blocking=True)
            else:
                dst = None if img is None else (img if frames == 'mapped' else True)
                e.env_step(self._flatten_action(action), sample_resets=(self.reset_mode == 'device'), frames=dst)
                if img is not None and frames == 'device':
                    img.copy_(e.frames, non_blocking=True)
                for v, dst in enumerate(more, 1):
                    if frames == 'mapped':
                        e.render(out=dst, view=v)
                    else:
                        dst.copy_(e.render(view=v), non_blocking=True)
                for m, dst in enumerate(masks):
                    if frames == 'mapped':
                        e.render_mask(out=dst, mask=m)
                    else:
                        dst.copy_(e.render_mask(mask=m), non_blocking=True)
                for r, dst in enumerate(rays):
                    if frames == 'mapped':
                        e.sense_rays(out=dst, sensor=r)
                    else:
                        dst.copy_(e.sense_rays(sensor=r), non_blocking=True)
                if spr is not None:
                    if frames == 'mapped':
                        e.observe_sprites(out=spr)
                    else:
                        spr.copy_(e.observe_sprites(), non_blocking=True)
            host.step_type.copy_(e.step_type, non_blocking=True)
            host.reward.copy_(e.reward, non_blocking=True)
            if host.discount is not None:
                host.discount.copy_(e.discount, non_blocking=True)
            main.synchronize()
            if auto:
                self._auto_record(frames, time.perf_counter() - t_begin)
            return host
        self.engine.env_step(self._flatten_action(action), sample_resets=(self.reset_mode == 'device'))
        if spr is not None:
            spr.copy_(e.observe_sprites(), non_blocking=True)
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=e.device)
            self._copy_events = [torch.cuda.Event() for _ in range(64)]
        copy = self._copy_stream
        host.step_type.copy_(e.step_type, non_blocking=True)
        host.reward.copy_(e.reward, non_blocking=True)
        if host.discount is not None:
            host.discount.copy_(e.discount, non_blocking=True)
        if self._image_key is not None or masks or rays:
            dsts = [host.observation[k] for k in self._image_keys]
            # a range of a view other than 0 or of a mask must start 16-byte aligned (moog_render_view,
            # moog_render_mask): one whose per-env bytes are not a multiple of 16 is drawn and copied
            # whole with the first range
            ranged = [v == 0 or e.view_buffer(v)[0].numel() % 16 == 0 for v in range(len(dsts))]
            mranged = [e.masks[m][0].numel() * 2 % 16 == 0 for m in range(len(masks))]
            rranged = [e.rays[r][0].numel() * 4 % 16 == 0 for r in range(len(rays))]
            chunks = max(1, min(int(chunks), len(self._copy_events), self.num_envs))
            # equal ranges: measured on B200 / PCIe 5 with 4096 64x64 frames, 4 equal ranges beat
            # 1, 2, 8 or 16 ranges and growing / shrinking ones (each render launch has a fixed
            # cost and does not fill the GPU when it is small)
            first = 0
            per = (self.num_envs + chunks - 1) // chunks
            for c in range(chunks):
                count = per
                count = min(count, self.num_envs - first)
                if count <= 0:
                    continue
                spans = []
                for v in range(len(dsts)):
                    span = (first, first + count) if ranged[v] else ((0, self.num_envs) if c == 0 else None)
                    if span is not None:
                        e.render(first=span[0], count=span[1] - span[0], view=v)
                        spans.append((v, span))
                mspans = []
                for m in range(len(masks)):
                    span = (first, first + count) if mranged[m] else ((0, self.num_envs) if c == 0 else None)
                    if span is not None:
                        e.render_mask(first=span[0], count=span[1] - span[0], mask=m)
                        mspans.append((m, span))
                rspans = []
                for r in range(len(rays)):
                    span = (first, first + count) if rranged[r] else ((0, self.num_envs) if c == 0 else None)
                    if span is not None:
                        e.sense_rays(first=span[0], count=span[1] - span[0], sensor=r)
                        rspans.append((r, span))
                ev = self._copy_events[c]
                ev.record(main)
                copy.wait_event(ev)
                with torch.cuda.stream(copy):
                    for v, (a, b) in spans:
                        dsts[v][a:b].copy_(e.view_buffer(v)[a:b], non_blocking=True)
                    for m, (a, b) in mspans:
                        masks[m][a:b].copy_(e.masks[m][a:b], non_blocking=True)
                    for r, (a, b) in rspans:
                        rays[r][a:b].copy_(e.rays[r][a:b], non_blocking=True)
                first += count
        copy.synchronize()
        main.synchronize()
        if auto:
            self._auto_record(frames, time.perf_counter() - t_begin)
        return host

    def host_pipeline(self, depth=2, frames='mapped'):
        """A `HostPipeline` over this environment: `submit(action)` / `collect()` with `depth`
        steps in flight, every TimeStep delivered in pinned host memory."""
        return HostPipeline(self, depth=depth, frames=frames)

    # frames='auto': kernel stores into the mapped host image hide the transfer behind the step
    # when the frames are small next to the step (4096 64x64 frames: 50 MB per 4.5 ms), but they
    # move fewer bytes per second over PCIe than the copy engines (16384 84x84 frames, 347 MB per
    # step: 986 k env-steps/s mapped, 1.48 M chunked).  The first calls try both and time them.
    _AUTO_TRIALS = 8

    def _auto_frames(self, img):
        if img is None or not img.is_pinned():
            return 'device'
        if self._auto_choice is not None:
            return self._auto_choice
        return ('mapped', 'chunked')[self._auto_calls % 2]

    def _auto_record(self, mode, seconds):
        if self._auto_choice is not None or mode not in self._auto_times:
            return
        self._auto_calls += 1
        if self._auto_calls > 2:                 # the first call of each mode warms up
            self._auto_times[mode].append(seconds)
        if self._auto_calls >= self._AUTO_TRIALS:
            best = {m: min(v) for m, v in self._auto_times.items() if v}
            self._auto_choice = min(best, key=best.get) if best else 'mapped'

    def observation(self):
        obs = {}
        for v, key in enumerate(self._image_keys):
            obs[key] = self.engine.render(view=v)
        for m, key in enumerate(self._mask_keys):
            obs[key] = self.engine.render_mask(mask=m)
        for r, key in enumerate(self._ray_keys):
            obs[key] = self.engine.sense_rays(sensor=r)
        if self._state_key is not None:
            obs[self._state_key] = self.engine.observe_sprites()
        return obs

    def _timestep(self, rendered=False):
        e = self.engine
        if rendered:
            # view 0 came with the step call; the other views are drawn behind it
            obs = {self._image_key: e.frames} if self._image_key is not None else {}
            for v, key in enumerate(self._image_keys[1:], 1):
                obs[key] = e.render(view=v)
            for m, key in enumerate(self._mask_keys):
                obs[key] = e.render_mask(mask=m)
            for r, key in enumerate(self._ray_keys):
                obs[key] = e.sense_rays(sensor=r)
            if self._state_key is not None:
                obs[self._state_key] = e.observe_sprites()
        else:
            obs = self.observation()
        return TimeStep(e.step_type, e.reward, e.discount, obs)

    def _flatten_action(self, action):
        if action is None:
            return None
        if isinstance(action, dict):
            cols = []
            for key, _, _, width in self.program.action_layout:
                a = action[key]
                a = a if torch.is_tensor(a) else torch.as_tensor(np.asarray(a))
                cols.append(a.to(self.engine.device, dtype=torch.float64).reshape(self.num_envs, width))
            return torch.cat(cols, dim=1)
        return action

    # -- extras -----------------------------------------------------------------
    def meta_state(self, env=0):
        """The env's meta_state as the dict the reference would hold (environment.py:129-131): the entries the
        program carries, strings decoded; None when the config has no meta_state."""
        prog = self.program
        if not getattr(prog, 'meta_vars', None):
            return None
        row = self.engine.state.envf[env].cpu().numpy()
        out = {}
        for key, slot in prog.meta_vars.items():
            v = float(row[slot])
            if isinstance(prog.meta_var_init.get(key), str) or key in getattr(prog, 'string_vars', ()):
                out[key] = prog.strings[int(v) - 1] if 1 <= int(v) <= len(prog.strings) else ''
            else:
                out[key] = int(v) if v == int(v) and abs(v) < 2 ** 53 else v
        return out

    def raise_errors(self):
        """Raises the data-dependent exceptions the reference would have raised."""
        err = self.engine.state.envi[:, 2]  # MOOG_EI_ERR
        bad = torch.nonzero(err).flatten()
        if bad.numel():
            i = int(bad[0])
            code = int(err[i])
            text = '; '.join(t for b, t in _ERR_TEXT.items() if code & b)
            raise ValueError('env {}: {}'.format(i, text))

    def state_dict(self):
        """Snapshot (cf. SimulationEnvironment, env_wrappers/simulation.py:55-83)."""
        return {k: getattr(self.engine.state, k).clone() for k in DeviceState.KEYS}

    def load_state_dict(self, sd):
        for k in DeviceState.KEYS:
            getattr(self.engine.state, k).copy_(sd[k])

    def episode_stats(self, reduce=True):
        """[sum reward, sum finished-episode length, finished episodes, env-steps];
        summed over ranks with one NCCL all_reduce when torch.distributed is up."""
        from . import dist as mdist
        s = self.engine.stats.clone()
        return mdist.reduce_stats(s) if reduce else s

    @property
    def action_dim(self):
        return max(self.program.action_dim, 1)


class HostPipeline(object):
    """Host-facing stepping with `depth` steps in flight (double buffering at depth 2).

    `step_to_host` hands the host one finished TimeStep per call and the GPU idles while the host
    looks at it (synchronise, Python, the next call's enqueue) -- and 8 ranks doing that against
    one host lose 20 % (round-1 scaling run).  Here the caller submits the action of step k+1
    BEFORE it collects the TimeStep of step k:

        pipe = env.host_pipeline(depth=2)
        pipe.submit(a0)
        for k in range(1, T):
            pipe.submit(a[k])          # enqueued behind step k-1, returns at once
            ts = pipe.collect()        # TimeStep of step k-1, in this slot's pinned host buffers
        ts = pipe.collect()

    i.e. the policy acts on an observation that is one step old (the usual actor pipeline); with
    depth 1 it is `step_to_host`.  Every submit copies that step's actions host -> device and
    every collect returns step_type / reward / discount / frames of every PILRenderer (and the
    RawState observation, the SpriteMasks and the RaySensors when the config has them) in pinned host
    memory, valid until `depth` further submits.  frames = 'mapped': the kernels store the frames, masks,
    rays and sprite observation
    straight into the slot's pinned buffers over PCIe; 'device': they are written to HBM and copied
    by a copy engine on a second stream while the next step runs.
    Reference protocol: moog/environment.py:98-126 (one `step` per submit, auto-reset included).
    """

    def __init__(self, env, depth=2, frames='mapped'):
        if depth < 1:
            raise ValueError('depth must be >= 1')
        if frames not in ('mapped', 'device'):
            raise ValueError("frames must be 'mapped' or 'device'")
        self.env, self.depth, self.frames = env, int(depth), frames
        e = env.engine
        self._main = torch.cuda.current_stream(e.device)
        self._copy = torch.cuda.Stream(device=e.device) if frames == 'device' else None
        n, ad = env.num_envs, env.action_dim
        pin = lambda *shape, dtype: torch.empty(shape, dtype=dtype).pin_memory()
        self._slots = []
        for _ in range(self.depth):
            spr = None
            obs = {}
            imgs = []  # one pinned image per view, in view order
            for v, key in enumerate(env._image_keys):  # pylint: disable=protected-access
                imgs.append(pin(*e.view_buffer(v).shape, dtype=torch.uint8))
                obs[key] = imgs[-1]
            if env._state_key is not None:  # pylint: disable=protected-access
                spr = obs[env._state_key] = pin(*e.sprites.shape, dtype=torch.float32)  # pylint: disable=protected-access
            masks = []  # one pinned mask per SpriteMask, in mask order
            for m, key in enumerate(env._mask_keys):  # pylint: disable=protected-access
                masks.append(pin(*e.masks[m].shape, dtype=torch.int16))
                obs[key] = masks[-1]
            rays = []  # one pinned reading per RaySensor, in sensor order
            for r, key in enumerate(env._ray_keys):  # pylint: disable=protected-access
                rays.append(pin(*e.rays[r].shape, dtype=torch.float32))
                obs[key] = rays[-1]
            self._slots.append(dict(
                ts=TimeStep(pin(n, dtype=torch.int32), pin(n, dtype=torch.float32), pin(n, dtype=torch.float32), obs),
                imgs=imgs, spr=spr, masks=masks, rays=rays,
                dev_masks=[torch.empty_like(d) for d in e.masks] if frames == 'device' else None,
                dev_rays=[torch.empty_like(d) for d in e.rays] if frames == 'device' else None,
                dev_imgs=[torch.empty_like(e.view_buffer(v)) for v in range(len(imgs))] if frames == 'device' else None,
                dev_sprites=(torch.empty_like(e.sprites) if (spr is not None and frames == 'device') else None),
                host_act=pin(n, ad, dtype=torch.float64),
                dev_act=torch.empty((n, ad), dtype=torch.float64, device=e.device),
                done=torch.cuda.Event(), stepped=torch.cuda.Event(), busy=False))
        self._head = 0     # next slot to submit into
        self._tail = 0     # next slot to collect
        self._in_flight = 0

    def submit(self, action=None):
        """Enqueue one `Environment.step(action)`; returns immediately."""
        if self._in_flight >= self.depth:
            raise RuntimeError('pipeline full: collect() a TimeStep before submitting another step')
        env, e = self.env, self.env.engine
        slot = self._slots[self._head]
        was_reset = not env._started  # pylint: disable=protected-access
        with torch.cuda.stream(self._main):
            if was_reset:
                env.reset()                                   # the first step of a MOOG env is its reset
                for v, img in enumerate(slot['imgs']):
                    img.copy_(e.view_buffer(v), non_blocking=True)
                if slot['spr'] is not None:
                    slot['spr'].copy_(e.sprites, non_blocking=True)
                for host_mask, dev in zip(slot['masks'], e.masks):
                    host_mask.copy_(dev, non_blocking=True)
                for host_rays, dev in zip(slot['rays'], e.rays):
                    host_rays.copy_(dev, non_blocking=True)
            else:
                act = None
                if action is not None:
                    action = env._flatten_action(action)  # pylint: disable=protected-access
                    if torch.is_tensor(action) and action.is_cuda:
                        slot['dev_act'].copy_(action.reshape(slot['dev_act'].shape), non_blocking=True)
                    else:
                        # staged in this slot's pinned buffer: the caller may reuse its own at once
                        slot['host_act'].copy_(torch.as_tensor(action).reshape(slot['host_act'].shape))
                        slot['dev_act'].copy_(slot['host_act'], non_blocking=True)
                    act = slot['dev_act']
                dsts = slot['imgs'] if self.frames == 'mapped' else slot['dev_imgs']
                e.env_step(act, sample_resets=(env.reset_mode == 'device'), frames=dsts[0] if dsts else None)
                for v in range(1, len(dsts)):
                    e.render(out=dsts[v], view=v)
                for m, dst in enumerate(slot['masks'] if self.frames == 'mapped' else slot['dev_masks']):
                    e.render_mask(out=dst, mask=m)
                for r, dst in enumerate(slot['rays'] if self.frames == 'mapped' else slot['dev_rays']):
                    e.sense_rays(out=dst, sensor=r)
                if slot['spr'] is not None:
                    e.observe_sprites(out=slot['spr'] if self.frames == 'mapped' else slot['dev_sprites'])
            ts = slot['ts']
            ts.step_type.copy_(e.step_type, non_blocking=True)
            ts.reward.copy_(e.reward, non_blocking=True)
            ts.discount.copy_(e.discount, non_blocking=True)
            if self.frames == 'device' and (slot['imgs'] or slot['masks'] or slot['rays'] or slot['spr'] is not None) \
                    and not was_reset:
                slot['stepped'].record(self._main)
                self._copy.wait_event(slot['stepped'])
                with torch.cuda.stream(self._copy):
                    for img, dev in zip(slot['imgs'], slot['dev_imgs']):
                        img.copy_(dev, non_blocking=True)
                    for host_mask, dev in zip(slot['masks'], slot['dev_masks']):
                        host_mask.copy_(dev, non_blocking=True)
                    for host_rays, dev in zip(slot['rays'], slot['dev_rays']):
                        host_rays.copy_(dev, non_blocking=True)
                    if slot['spr'] is not None:
                        slot['spr'].copy_(slot['dev_sprites'], non_blocking=True)
                    slot['done'].record(self._copy)
            else:
                slot['done'].record(self._main)
        slot['busy'] = True
        self._head = (self._head + 1) % self.depth
        self._in_flight += 1

    def collect(self):
        """The oldest submitted step's TimeStep (host tensors), once all of it has arrived."""
        if self._in_flight == 0:
            raise RuntimeError('nothing in flight')
        slot = self._slots[self._tail]
        slot['done'].synchronize()
        slot['busy'] = False
        self._tail = (self._tail + 1) % self.depth
        self._in_flight -= 1
        return slot['ts']

    def last_event(self):
        """CUDA event of the most recently submitted step's completion (for device-side timing)."""
        return self._slots[(self._head - 1) % self.depth]['done']

    def step(self, action=None):
        """submit + collect at depth 1 semantics: the TimeStep of THIS action (drains the pipeline first)."""
        while self._in_flight:
            self.collect()
        self.submit(action)
        return self.collect()
