"""Renderer spec with PILRenderer's constructor (pil_renderer.py:37-86).

The frames are produced by the sm_100a rasteriser, which reproduces Pillow's
polygon fill / alpha blend / Lanczos down-sampling bit for bit; Pillow itself
is not used on this path.
"""

import abc

from . import color_maps
from . import polygon_modifiers


class AbstractObserver(abc.ABC):
    def observation_spec(self):
        return self._observation_spec


class _ImageSpec(object):
    def __init__(self, shape):
        import numpy as np
        self.shape = shape
        self.dtype = np.dtype(np.uint8)


class PILRenderer(AbstractObserver):
    def __init__(self, image_size=(64, 64), anti_aliasing=1, bg_color=None,
                 color_to_rgb=None, polygon_modifier=None):
        self._image_size = tuple(image_size)
        self._anti_aliasing = anti_aliasing
        self._canvas_size = (anti_aliasing * image_size[0],
                             anti_aliasing * image_size[1])
        if polygon_modifier is None:
            polygon_modifier = polygon_modifiers.DoNothing()
        self._polygon_modifier = polygon_modifier
        if isinstance(color_to_rgb, str):
            color_to_rgb = getattr(color_maps, color_to_rgb)
        self.color_to_rgb = color_to_rgb
        self._bg_color = (0, 0, 0) if bg_color is None else tuple(bg_color)
        self._observation_spec = _ImageSpec(self._image_size + (3,))

    @property
    def polygon_modifier(self):
        return self._polygon_modifier


class RawState(AbstractObserver):
    """Marker observer for the sprites' state (raw_state.py:17-19).  Instead of an OrderedDict of
    layer -> list of Sprite, the batched environment returns under this key one float32 tensor
    [num_envs, S, 16] over all S sprite slots of the record, in layer order and, within a layer, in
    list (z-) order.  Columns: x, y, shape id, angle, scale, aspect_ratio, c0, c1, c2, opacity,
    x_vel, y_vel, angle_vel, mass, the slot's layer index, alive (1 for a live sprite; every other
    column of an empty slot is 0).  `BatchedEnvironment.shape_names()` names the shape ids."""

    _observation_spec = None
