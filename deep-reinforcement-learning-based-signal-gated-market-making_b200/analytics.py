"""StrategyAnalytics (analytics/mm_analyzer.py:5-56) as device reductions.

``StrategyAnalytics(df)`` keeps the reference's properties and ``summary_dict``; ``population_summary`` does the
same for a whole batch of traces in one launch (one warp per trace), and ``backtest_population`` traces a whole population
and summarises it without leaving the device.  The float64 reductions follow pandas /
numpy's pairwise summation order, so every figure -- the trade Sharpe ratio included -- is bit-identical to the
reference's.  Plotting (BacktestVisualizer) is out of scope.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib

KEYS = ("Total PnL", "MAP (Risk)", "PnLMAP (Eff)", "Max DD", "Sharpe", "Trades")


def population_summary(wealth, inventory, is_trade, device=None):
    """``wealth`` float64 [B, T], ``inventory`` int [B, T], ``is_trade`` bool [B, T] -> float64 [B, 6] in KEYS order."""
    if device is None:
        device = torch.cuda.current_device()
    w = np.ascontiguousarray(np.atleast_2d(wealth), np.float64)
    iv = np.ascontiguousarray(np.atleast_2d(inventory), np.int32)
    tr = np.ascontiguousarray(np.atleast_2d(np.asarray(is_trade)).astype(bool), np.uint8)
    if not (w.shape == iv.shape == tr.shape):
        raise ValueError("wealth, inventory and is_trade must have the same [traces, steps] shape")
    B, T = w.shape
    out = np.zeros((B, 6), np.float64)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    p = (lambda a: C.c_void_p(a.ctypes.data) if a.size else None)
    _lib.check(_lib.lib().sgmm_trace_analytics_host(B, T, p(w), p(iv), p(tr), C.c_void_p(out.ctypes.data), int(device), st))
    return out


def backtest_population(bundle, genomes=None, adv_genomes=None, *, master=None, count=None, sigma=None, seed=None, generation=0,
                        first_index=0, adv_master=None, adv_sigma=None, phi, fee_rate=0.0, hidden=32):
    """Backtest and risk analytics of a whole population: the population arguments of
    :func:`engine.rollout_trace_population` -> ``(fitness float64[P], trades int32[P], summary float64[P, 6])``, CUDA
    tensors, summary columns in ``KEYS`` order.  Row i equals
    ``StrategyAnalytics(StrategyRecorder.from_trace(rollout_trace(...)[2], bundle).to_dataframe()).summary_dict`` of
    individual i.  Only wealth, inventory and the fills are traced; nothing goes through the host."""
    from .engine import rollout_trace_population, _stream
    fit, trd, cols = rollout_trace_population(bundle, genomes, adv_genomes, master=master, count=count, sigma=sigma, seed=seed,
                                              generation=generation, first_index=first_index, adv_master=adv_master,
                                              adv_sigma=adv_sigma, phi=phi, fee_rate=fee_rate, hidden=hidden,
                                              columns=("wealth", "inventory", "fill_buy", "fill_sell"))
    P, T = cols["wealth"].shape
    out = torch.empty(P, 6, dtype=torch.float64, device=fit.device)
    if P == 0:
        return fit, trd, out
    is_trade = (cols["fill_buy"] | cols["fill_sell"]).to(torch.uint8)          # the recorder's is_trade: fill_buy or fill_sell
    scratch = torch.empty(P, T, dtype=torch.float64, device=fit.device)
    p = (lambda x: x.data_ptr() if x.numel() else None)
    _lib.check(_lib.lib().sgmm_trace_analytics(P, T, p(cols["wealth"]), None, None, p(cols["inventory"]), p(is_trade),
                                               p(scratch), out.data_ptr(), _stream(bundle.device)))
    return fit, trd, out


class StrategyAnalytics:
    """Drop-in for analytics/mm_analyzer.py:5-56 (same constructor argument, properties and ``summary_dict``)."""

    def __init__(self, df, device=None):
        self.df = df
        s = population_summary(np.asarray(df['wealth'], np.float64), np.asarray(df['inventory']),
                               np.asarray(df['is_trade']).astype(bool), device)[0]
        self._s = s

    total_pnl = property(lambda self: float(self._s[0]))
    mean_absolute_position = property(lambda self: float(self._s[1]))
    pnl_to_map_ratio = property(lambda self: float(self._s[2]))
    max_drawdown = property(lambda self: float(self._s[3]))
    sharpe_ratio = property(lambda self: float(self._s[4]))

    @property
    def summary_dict(self) -> dict:
        return {'Total PnL': self.total_pnl, 'MAP (Risk)': self.mean_absolute_position,
                'PnLMAP (Eff)': self.pnl_to_map_ratio, 'Max DD': self.max_drawdown,
                'Sharpe': self.sharpe_ratio, 'Trades': int(self._s[5])}
