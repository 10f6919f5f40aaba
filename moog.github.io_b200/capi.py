"""ctypes binding of libmoog_b200.so (include/moog_b200.h).

The library is the product path: there is no CPU or PyTorch fallback.  If it
is missing it is built with nvcc (moog_b200.build); if that fails, importing
this module raises.
"""
import ctypes
import os

from . import build as _build

_lib = None


class MoogState(ctypes.Structure):
    """`moog_state`: device pointers to the SoA state record."""
    _fields_ = [('dyn', ctypes.c_void_p), ('stat', ctypes.c_void_p),
                ('meta', ctypes.c_void_p), ('cnt', ctypes.c_void_p),
                ('envi', ctypes.c_void_p), ('envf', ctypes.c_void_p),
                ('vtx', ctypes.c_void_p)]


class MoogStepIO(ctypes.Structure):
    """`moog_step_io`."""
    _fields_ = [('actions', ctypes.c_void_p), ('noise', ctypes.c_void_p),
                ('rule_noise', ctypes.c_void_p),
                ('pool', ctypes.POINTER(MoogState)),
                ('pool_size', ctypes.c_int32),
                ('reset_index', ctypes.c_void_p), ('seed', ctypes.c_uint64),
                ('reward', ctypes.c_void_p), ('step_type', ctypes.c_void_p),
                ('discount', ctypes.c_void_p), ('counters', ctypes.c_void_p),
                ('stats', ctypes.c_void_p), ('sample_resets', ctypes.c_int32),
                ('frames', ctypes.c_void_p)]


class MoogRaySpec(ctypes.Structure):
    """`moog_ray_spec`."""
    _fields_ = [('agent_layer', ctypes.c_int32), ('agent_index', ctypes.c_int32),
                ('layers', ctypes.c_uint32), ('n_rays', ctypes.c_int32),
                ('max_range', ctypes.c_double), ('dirs', ctypes.c_void_p)]


# every symbol include/moog_b200.h declares
SYMBOLS = ('moog_program_create', 'moog_program_destroy',
           'moog_program_env_smem_bytes', 'moog_env_step',
           'moog_env_post_reset', 'moog_physics_step', 'moog_overlap_pairs',
           'moog_render', 'moog_strerror', 'moog_last_cuda_error',
           'moog_launch_count', 'moog_host_paths_overlap',
           'moog_host_points_in_path', 'moog_step_launch_info',
           'moog_step_draws_frames', 'moog_program_set_option',
           'moog_program_validate', 'moog_observe_sprites', 'moog_render_view',
           'moog_render_plan', 'moog_render_mask', 'moog_mask_plan', 'moog_ray_sensor')


# include/moog_b200.h return codes
E_INVAL, E_CUDA, E_TOO_BIG, E_UNSUPPORTED = -1, -2, -3, -4


class MoogError(RuntimeError):
    pass


def lib_path():
    return _build.LIB


def lib():
    """Loads (building first when needed) the CUDA library."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if _build.is_stale():
        try:
            _build.build()
        except Exception as exc:  # pylint: disable=broad-except
            if not os.path.exists(path):
                raise MoogError(
                    'libmoog_b200.so is missing and could not be built ({}); '
                    'the device path has no fallback'.format(exc))
    L = ctypes.CDLL(path)
    vp, ci = ctypes.c_void_p, ctypes.c_int
    L.moog_program_create.argtypes = [vp, ctypes.c_size_t, ctypes.POINTER(vp)]
    L.moog_program_create.restype = ci
    L.moog_program_destroy.argtypes = [vp]
    L.moog_program_destroy.restype = None
    L.moog_program_env_smem_bytes.argtypes = [vp]
    L.moog_program_env_smem_bytes.restype = ci
    L.moog_env_step.argtypes = [vp, ctypes.POINTER(MoogState), ci,
                                ctypes.POINTER(MoogStepIO), vp]
    L.moog_env_step.restype = ci
    L.moog_env_post_reset.argtypes = [vp, ctypes.POINTER(MoogState), ci, vp, vp]
    L.moog_env_post_reset.restype = ci
    L.moog_physics_step.argtypes = [vp, ctypes.POINTER(MoogState), ci, vp, vp, vp]
    L.moog_physics_step.restype = ci
    L.moog_overlap_pairs.argtypes = [vp, ctypes.POINTER(MoogState), ci, ci, ci, vp, vp]
    L.moog_overlap_pairs.restype = ci
    L.moog_render.argtypes = [vp, ctypes.POINTER(MoogState), ci, vp, vp]
    L.moog_render.restype = ci
    L.moog_observe_sprites.argtypes = [vp, ctypes.POINTER(MoogState), ci, vp, vp]
    L.moog_observe_sprites.restype = ci
    L.moog_render_view.argtypes = [vp, ctypes.POINTER(MoogState), ci, ci, vp, vp]
    L.moog_render_view.restype = ci
    L.moog_strerror.argtypes = [ci]
    L.moog_strerror.restype = ctypes.c_char_p
    L.moog_last_cuda_error.argtypes = []
    L.moog_last_cuda_error.restype = ctypes.c_char_p
    L.moog_host_paths_overlap.argtypes = [vp, ci, vp, ci]
    L.moog_host_paths_overlap.restype = ci
    L.moog_host_points_in_path.argtypes = [vp, ci, vp, ci, vp]
    L.moog_host_points_in_path.restype = None
    L.moog_step_launch_info.argtypes = [vp, ci, ctypes.POINTER(ci), ctypes.POINTER(ci), ctypes.POINTER(ci)]
    L.moog_step_launch_info.restype = ci
    L.moog_step_draws_frames.argtypes = [vp, ci]
    L.moog_step_draws_frames.restype = ci
    L.moog_program_set_option.argtypes = [vp, ctypes.c_char_p, ci]
    L.moog_program_set_option.restype = ci
    L.moog_program_validate.argtypes = [vp, ctypes.c_size_t]
    L.moog_program_validate.restype = ci
    L.moog_render_plan.argtypes = [vp, ctypes.c_size_t, ci, ctypes.POINTER(ci), ctypes.POINTER(ci)]
    L.moog_render_plan.restype = ci
    L.moog_render_mask.argtypes = [vp, ctypes.POINTER(MoogState), ci, ci, vp, vp]
    L.moog_render_mask.restype = ci
    L.moog_mask_plan.argtypes = [vp, ctypes.c_size_t, ci, ctypes.POINTER(ci), ctypes.POINTER(ci)]
    L.moog_mask_plan.restype = ci
    L.moog_ray_sensor.argtypes = [vp, ctypes.POINTER(MoogState), ci, ctypes.POINTER(MoogRaySpec), vp, vp]
    L.moog_ray_sensor.restype = ci
    L.moog_launch_count.argtypes = []
    L.moog_launch_count.restype = ctypes.c_int64
    _lib = L
    return L


def check(code):
    if code != 0:
        L = lib()
        msg = L.moog_strerror(code).decode()
        if code == E_CUDA:
            msg += ': ' + L.moog_last_cuda_error().decode()
        raise MoogError('libmoog_b200: {} ({})'.format(msg, code))


def launch_count():
    return int(lib().moog_launch_count())


def render_plan(blob, view=0):
    """How the render kernel draws view `view` of a program blob, without a device
    (include/moog_b200.h moog_render_plan): (code, chunk_rows, smem_bytes); code 0, or
    E_UNSUPPORTED for a view no chunk size can hold, or E_INVAL."""
    buf = ctypes.create_string_buffer(bytes(blob), len(blob))
    rows, smem = ctypes.c_int(), ctypes.c_int()
    code = int(lib().moog_render_plan(buf, len(blob), int(view), ctypes.byref(rows), ctypes.byref(smem)))
    return code, rows.value, smem.value


def mask_plan(blob, mask=0):
    """How the mask kernel draws mask `mask` of a program blob, without a device
    (include/moog_b200.h moog_mask_plan): (code, band_rows, smem_bytes); code 0, or
    E_UNSUPPORTED for a mask no band can hold, or E_INVAL."""
    buf = ctypes.create_string_buffer(bytes(blob), len(blob))
    rows, smem = ctypes.c_int(), ctypes.c_int()
    code = int(lib().moog_mask_plan(buf, len(blob), int(mask), ctypes.byref(rows), ctypes.byref(smem)))
    return code, rows.value, smem.value


class DeviceProgram(object):
    """Owns a `moog_program*`."""

    def __init__(self, blob):
        self._h = ctypes.c_void_p()
        buf = ctypes.create_string_buffer(bytes(blob), len(blob))
        check(lib().moog_program_create(buf, len(blob), ctypes.byref(self._h)))

    @property
    def handle(self):
        return self._h

    def env_smem_bytes(self):
        return int(lib().moog_program_env_smem_bytes(self._h))

    def step_launch_info(self, n_envs):
        """(envs resident per SM, warps per env, shared-memory bytes per env)."""
        r, w, s = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        check(lib().moog_step_launch_info(self._h, int(n_envs), ctypes.byref(r), ctypes.byref(w), ctypes.byref(s)))
        return r.value, w.value, s.value

    def step_draws_frames(self, n_envs):
        """Whether `moog_env_step` with frames draws them inside the step kernel."""
        r = int(lib().moog_step_draws_frames(self._h, int(n_envs)))
        if r < 0:
            check(r)
        return bool(r)

    def set_option(self, name, value):
        """One launch option of this program (include/moog_b200.h moog_program_set_option)."""
        check(lib().moog_program_set_option(self._h, name.encode(), int(value)))

    def close(self):
        if self._h:
            lib().moog_program_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # pylint: disable=broad-except
            pass
