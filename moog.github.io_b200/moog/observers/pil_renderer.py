"""Renderer spec with PILRenderer's constructor (pil_renderer.py:37-86).

The frames are produced by the sm_100a rasteriser, which reproduces Pillow's
polygon fill / alpha blend / Lanczos down-sampling bit for bit; Pillow itself
is not used on this path.
"""

import abc
import math

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


class RaySensor(AbstractObserver):
    """Range finder: rays from an agent sprite to the first outline they cross.  The reference has no such
    observer; this one is an extension.

    The batched environment returns under this key one float32 tensor [num_envs, num_rays, 2].
    - Origin o: the position (x, y) of sprite `agent_index` of layer `agent_layer`.  When that layer holds
      fewer live sprites, every ray reads "no hit".
    - Ray k points along phi_k = direction - fov / 2 + fov * (k + 0.5) / num_rays, counter-clockwise from +x
      in the world frame: the rays do not turn with the agent (FirstPersonAgent only translates either).
      The host computes d_k = (np.cos(phi_k), np.sin(phi_k)) once, in float64 (`directions()`); the device
      evaluates no trigonometric function.
    - Targets: every live sprite of `layers` (None: all layers) except the agent itself, whatever its
      opacity.  A sprite's outline is the closed polygon through its cached world vertices; vertex j is
      joined to vertex (j + 1) mod nv, and a degenerate edge never hits.
    - Hit distance, float64, evaluated as written (a x b = a.x * b.y - a.y * b.x): for an edge (a, b),
      e = b - a, w = a - o, den = d x e; when den != 0, t = (w x e) / den and u = (w x d) / den, and the
      edge is hit when 0 <= u <= 1 and t >= 0.  A sprite's t is its smallest edge t, or 0 when o lies
      inside its outline by the even-odd rule (edges with (a.y > o.y) != (b.y > o.y) and
      o.x < a.x + (o.y - a.y) * (b.x - a.x) / (b.y - a.y)).
    - Reading of ray k: the smallest t over the targets, a tie going to the later sprite in draw order.
      When t <= max_range it is (float32(t / max_range), float32(slot)), the slot being the RawState row
      (`program.layer_off` maps it to its layer); otherwise (1.0, -1.0).
    Rays do not wrap under TorusGeometry.  Limits: 1 <= num_rays <= 256, a finite max_range > 0,
    0 < fov <= 2 pi, at most 8 RaySensors per config."""

    def __init__(self, agent_layer, num_rays=32, max_range=0.5, fov=2 * math.pi, direction=math.pi / 2,
                 layers=None, agent_index=0):
        self._agent_layer = agent_layer
        self._num_rays = num_rays
        self._max_range = max_range
        self._fov = fov
        self._direction = direction
        self._layers = None if layers is None else list(layers)
        self._agent_index = agent_index
        self._observation_spec = None

    def directions(self):
        """[num_rays, 2] float64: (cos phi_k, sin phi_k) of every ray."""
        import numpy as np
        k = np.arange(int(self._num_rays), dtype=np.float64)
        phi = self._direction - self._fov / 2 + self._fov * (k + 0.5) / self._num_rays
        return np.stack([np.cos(phi), np.sin(phi)], axis=1)
