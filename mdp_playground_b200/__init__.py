"""mdp_playground_b200: B200-native batched RLToyEnv step path.

`VectorRLToyEnv` mirrors the reference's `RLToyEnv` constructor keys and
reset/step semantics and runs every step on hand-written sm_100a CUDA kernels
(libmdpp_b200.so, C ABI in include/mdpp_b200.h).  No CPU fallback.
"""
from .vector_env import VectorRLToyEnv  # noqa: F401
from .wrapper_tail import VectorGymEnvTail  # noqa: F401
from .qlearning import GridQLearner, TabularQLearner  # noqa: F401
from .ars import LinearARS  # noqa: F401

__all__ = ["VectorRLToyEnv", "VectorGymEnvTail", "TabularQLearner", "GridQLearner",
           "LinearARS"]
__version__ = "0.1.0"
