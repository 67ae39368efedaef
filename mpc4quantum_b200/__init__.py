"""mpc4quantum_b200: the receding-horizon loop of andgoldschmidt/MPC4quantum on B200 (sm_100a).

Same module layout and names as the reference package (mpc4quantum/__init__.py:3-7 star-imports experiment,
linearize, model, mpc, vectorize); the arithmetic runs in libm4q.so (csrc/, C ABI in include/m4q.h).
"""
from .experiment import *   # noqa: F401,F403
from .linearize import *    # noqa: F401,F403
from .model import *        # noqa: F401,F403
from .mpc import *          # noqa: F401,F403
from .vectorize import *    # noqa: F401,F403
from . import experiment, linearize, model, optimize, vectorize  # noqa: F401  (`mpc` names the function, as upstream)
from ._lib import supported_shapes  # noqa: F401

__version__ = '0.1.0'
