"""sgmm_b200 -- B200-native population rollout of the signal-gated market-making MDP.

Drop-in for the hot path of KAS-W/Deep-Reinforcement-Learning-Based-Signal-Gated-Market-Making:
``FTPEnv`` (Env/market_env.py), ``evaluate_individual`` / ``DRLEngine`` (Env/drl_engine.py),
``TradingPolicy`` / ``AdversaryPolicy`` / ``NeuroEvolution`` (models/model.py) and a
``StrategyRecorder`` (Env/recorder.py) fed by the device trace.  All compute goes through the
C ABI of ``libsgmm_b200.so`` (include/sgmm.h, hand-written sm_100a CUDA); there is no CPU fallback.
"""
from ._lib import SgmmError, SgmmLibraryError, lib  # noqa: F401
from .env import FTPEnv  # noqa: F401
from .policy import AdversaryPolicy, NeuroEvolution, TradingPolicy, genome_len  # noqa: F401
from .bundle import Bundle, normalise, bundle_windows, day_bundle, concat_days  # noqa: F401
from .analytics import StrategyAnalytics, backtest_population, population_summary  # noqa: F401
from .engine import (DRLEngine, DeviceGA, DeviceGASweep, evaluate_individual, rollout_population, rollout_population_async, rollout_seeded,  # noqa: F401
                     rollout_trace, rollout_trace_population, rollout_table, rollout_spec256_audit, rollout_tc_audit, measure_fp32_peak)
from .recorder import StrategyRecorder  # noqa: F401
from .benchmarks import FOICPolicy, GLFTPolicy  # noqa: F401
from . import synthetic  # noqa: F401

__version__ = "0.1.1"
