"""B200-native batched simulator for the per-step hot path of Layered-Safe-MARL's
`navigation_graph_safe` environment (see DESIGN.md). The compute path is the sm_100a library
`liblsm_b200.so` behind include/lsm_b200.h; there is no CPU fallback."""
from .config import (AirTaxiConfig, DoubleIntegratorConfig, RewardBinaryConfig, RewardWeightConfig,
                     ScenarioParams, scenario_params_from_args)
from .vec_env import B200GraphDummyVecEnv, B200GraphVecEnv
from .rollout import DeviceGraphRolloutBuffer
from .safety_filter import SafetyFilter
from . import eval_scenarios

__all__ = ['AirTaxiConfig', 'DoubleIntegratorConfig', 'RewardBinaryConfig', 'RewardWeightConfig',
           'ScenarioParams', 'scenario_params_from_args', 'B200GraphVecEnv', 'B200GraphDummyVecEnv',
           'DeviceGraphRolloutBuffer', 'SafetyFilter', 'eval_scenarios']
