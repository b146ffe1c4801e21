"""xline_b200 -- B200-native implementation of xline's ``Line.track`` particle push.

Public API mirrors the reference (``xline/__init__.py:10-21``): ``Line``, ``Particles``
and the element classes.  The arithmetic runs in hand-written sm_100a CUDA kernels behind
the C ABI of ``include/xline_b200.h`` (``libxline_b200.so``); there is no CPU fallback.
"""
__version__ = "0.1.0"

from . import elements
from .elements import *  # noqa: F401,F403
from .line import Line
from .moments import BeamMoments, beam_moments
from .particles import Particles
from .tangent import (ClosedOrbit, Envelope, RadiationEquilibrium, TangentMap, closed_orbit,
                      radiation_equilibrium)
from .tunes import monitor_tunes, naff

XlineTestParticles = Particles  # the reference's name (xline/particles.py:4)

__all__ = list(elements.__all__) + ["Line", "Particles", "XlineTestParticles", "elements", "BeamMoments",
                                    "beam_moments", "naff", "monitor_tunes", "TangentMap", "closed_orbit",
                                    "ClosedOrbit", "Envelope", "radiation_equilibrium", "RadiationEquilibrium"]
