"""Expression compiler: skill -> scalar programs (lower.py) -> CUDA translation unit (emit.py)."""
from .lower import PinvProgram, QpProgram, NlpProgram  # noqa: F401
from .emit import emit_skill, Emitter, emit_c_function  # noqa: F401
