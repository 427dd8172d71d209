"""Importable alias of the `steered-mixture-of-experts_b200/` package directory.

The product package directory carries the reference's name (with a hyphen, so it is not a
Python identifier); this stub makes it importable as `smoe_b200` by pointing its module search
path at that directory.  All code lives there.
"""
import os as _os

_pkg_dir = _os.path.join(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))),
                         "steered-mixture-of-experts_b200")
__path__.insert(0, _pkg_dir)

from .smoe import Smoe, AdamOptimizer, sliding_window  # noqa: E402,F401
from .quantizer import quantize_params, rescaler        # noqa: E402,F401
from .utils import reduce_params, save_model, load_params, read_image, write_image, psnr  # noqa: E402,F401
from . import smoe_reconstruction, smoe_reconstruction_decoded, smoe_test  # noqa: E402,F401
from .render import SmoePointRenderer, SmoeRenderer  # noqa: E402,F401
