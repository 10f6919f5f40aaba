"""Observer specs (reference: moog/observers/)."""

from . import color_maps
from . import polygon_modifiers
from .pil_renderer import AbstractObserver
from .pil_renderer import PILRenderer
from .pil_renderer import RawState
from .pil_renderer import RaySensor
from .pil_renderer import SpriteMask
