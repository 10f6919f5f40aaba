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


class SpriteMask(AbstractObserver):
    """Which sprite each pixel shows.  The reference has no such observer; this one is an extension.

    The batched environment returns under this key one int16 tensor [num_envs, H, W] for
    `image_size=(W, H)` (PILRenderer's order).  For output pixel mask[n, j, x], let y = H - 1 - j
    (the frames' np.flipud).  The value is the record slot s of the LAST sprite in draw order whose
    polygon covers canvas pixel (x, y), or -1 where no sprite does.
    - "Covers" means covered by the fill the frames use: Pillow's ImageDraw.Draw(canvas, 'RGBA')
      .polygon (polygon_generic with deferred horizontal edges).  The vertices are the int-truncated
      world vertices times the image size, after `polygon_modifier`.
    - Draw order is slot order over the live slots (layer order, then list order).
    - Only sprites whose ink alpha byte uint8(int64(opacity)) is non-zero count: a sprite with alpha
      0 is invisible in the frames and absent from the mask.
    - Every TorusGeometry copy of slot s writes s.
    The slot is the RawState row, so state[n, mask[n, j, x]] is the sprite shown at that pixel.  A
    mask is scan-converted at image_size: no anti-aliasing, no colours, no background."""

    def __init__(self, image_size=(64, 64), polygon_modifier=None):
        self._image_size = tuple(image_size)
        if polygon_modifier is None:
            polygon_modifier = polygon_modifiers.DoNothing()
        self._polygon_modifier = polygon_modifier
        self._observation_spec = None

    @property
    def polygon_modifier(self):
        return self._polygon_modifier
