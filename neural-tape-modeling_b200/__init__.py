"""ntm_b200 -- B200-native engine for the recurrent forward pass of neural-tape-modeling
(GRU-HS[64] tape nonlinearity, DiffDelGRU delay line).  See DESIGN.md."""
from . import driver, lib, sharding, signals  # noqa: F401
from .losses import DCPreESR, ESRLoss, MultiResolutionSTFTLoss  # noqa: F401
from .model import (RNN, BlockStream, DelayBlockStream, DiffDelRNN, RealtimeDelayStream, RealtimeStream,  # noqa: F401
                    TimeVaryingDelayLine)

__all__ = ["RNN", "BlockStream", "RealtimeStream", "DiffDelRNN", "DelayBlockStream", "RealtimeDelayStream", "TimeVaryingDelayLine", "ESRLoss", "DCPreESR", "MultiResolutionSTFTLoss", "driver", "lib", "sharding", "signals"]
