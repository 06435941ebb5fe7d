"""tobac_flow_b200 — B200-native (sm_100a) dense-flow hot path behind the ``tobac_flow.flow.Flow`` API."""
from .flow import (Flow, create_flow, calculate_flow, calculate_flow_2, smooth_flow_step, pair_to_8bit,  # noqa: F401
                   NativeError, operand_cache_clear)
from .dis import DISOpticalFlow  # noqa: F401

__all__ = ["Flow", "create_flow", "calculate_flow", "calculate_flow_2", "smooth_flow_step", "pair_to_8bit",
           "NativeError", "operand_cache_clear", "DISOpticalFlow"]
