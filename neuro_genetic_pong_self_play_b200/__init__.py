"""B200-native population-evaluation hot path of n00b001/neuro-genetic-pong-self-play.

Host side in Python (like the reference), compute in hand-written sm_100a CUDA kernels behind the
C ABI of libngp.so (include/ngp.h).  No CPU fallback exists: Engine raises without a CUDA device or
when the library cannot be built/loaded."""
from . import _lib
from ._lib import (ACT_DOWN, ACT_NONE, ACT_UP, CORE_INTERPRETER, CORE_TRANSLATED, OPP_HARDCODED, OPP_ROBOT, OPP_SCORE_HARDCODED,
                   PLAYER_EXTERNAL, SCHEDULE_REFERENCE, SCHEDULE_ROUND_ROBIN, STATE_START_1P, STATE_START_2P, NgpError)
from .config import Config
from .engine import Engine, load_rom

__all__ = ["Engine", "Config", "NgpError", "load_rom", "ACT_NONE", "ACT_UP", "ACT_DOWN", "STATE_START_1P", "STATE_START_2P",
           "SCHEDULE_REFERENCE", "SCHEDULE_ROUND_ROBIN", "CORE_INTERPRETER", "CORE_TRANSLATED", "OPP_HARDCODED", "OPP_SCORE_HARDCODED",
           "OPP_ROBOT", "PLAYER_EXTERNAL"]
