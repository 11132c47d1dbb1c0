"""casclik_b200 — B200-native batched CLIK controller-step engine with CASCLIK's Python API.

    import casclik_b200 as cc
    from casclik_b200 import cs          # stands in for `import casadi as cs`

Exports mirror reference casclik/__init__.py:1-7 (constraint classes, SkillSpecification,
PseudoInverseController, ReactiveQPController, ReactiveNLPController).  The reference's
ModelPredictiveController (an NLP over a horizon with nonlinear dynamics) is out of scope
(SURVEY.md §2 row 6).
"""
from . import sym as cs  # noqa: F401
from .constraints import *  # noqa: F401,F403
from .skill_specification import SkillSpecification  # noqa: F401
from .controllers import PseudoInverseController, ReactiveQPController, ReactiveNLPController  # noqa: F401
from . import fk  # noqa: F401

__version__ = "0.1.0"
