from .pseudo_inverse import PseudoInverseController  # noqa: F401
from .reactive_qp import ReactiveQPController  # noqa: F401
from .reactive_nlp import ReactiveNLPController  # noqa: F401
