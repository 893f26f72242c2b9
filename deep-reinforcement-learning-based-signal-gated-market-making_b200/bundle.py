"""Device-resident bundles.

The reference passes a 7-tuple of host arrays ``(s1, s2, mid_next, best_ask, best_bid, buy_max,
sell_min)`` (pipeline/agent_trainer.py:75-77) plus ``train_stats`` into every rollout
(Env/drl_engine.py:9-11).  ``Bundle`` normalises the signals with the caller's own numpy
expression (drl_engine.py:33-34), uploads everything once and runs the prologue kernel that
derives the integer fill thresholds (include/sgmm.h, sgmm_bundle_create).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib


def normalise(bundle, train_stats):
    """``(s[t]-m)/s`` evaluated element-wise in the caller's dtypes (NEP-50 promotion is the same
    for the vectorised and the scalar expression), then the float32 cast that
    ``torch.tensor(..., dtype=torch.float32)`` applies (drl_engine.py:33-35)."""
    s1, s2 = np.asarray(bundle[0]), np.asarray(bundle[1])
    z1 = ((s1 - train_stats['s1_m']) / train_stats['s1_s']).astype(np.float32)
    z2 = ((s2 - train_stats['s2_m']) / train_stats['s2_s']).astype(np.float32)
    return z1, z2


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a.size else None


class Bundle:
    """Handle of a ``sgmm_bundle`` living on one CUDA device."""

    def __init__(self, z1, z2, mid_next, best_ask, best_bid, buy_max, sell_min, tick_size,
                 device=None, stream=None):
        if device is None:
            device = torch.cuda.current_device()
        self.device = int(torch.device(device).index if not isinstance(device, int) else device)
        arrs = [np.ascontiguousarray(z1, np.float32), np.ascontiguousarray(z2, np.float32)]
        arrs += [np.ascontiguousarray(a, np.float64) for a in (mid_next, best_ask, best_bid, buy_max, sell_min)]
        n = arrs[0].size
        if any(a.ndim != 1 or a.size != n for a in arrs):
            raise ValueError("bundle arrays must be 1-D and of equal length")
        self.T = int(n)
        self.tick_size = float(tick_size)
        self._h = C.c_void_p()
        st = C.c_void_p(stream if stream is not None else torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(_lib.lib().sgmm_bundle_create(C.byref(self._h), self.T, *[_ptr(a) for a in arrs],
                                                 self.tick_size, self.device, st))

    @classmethod
    def from_arrays(cls, bundle, train_stats, tick_size, device=None):
        """From the reference's 7-tuple + ``train_stats`` dict (keys s1_m, s1_s, s2_m, s2_s)."""
        z1, z2 = normalise(bundle, train_stats)
        return cls(z1, z2, bundle[2], bundle[3], bundle[4], bundle[5], bundle[6], tick_size, device)

    @property
    def handle(self):
        if not self._h:
            raise RuntimeError("bundle is closed")
        return self._h

    def thresholds(self):
        """(Ka, Kb) int32[T]: fill_sell <=> off_a <= Ka, fill_buy <=> off_b <= Kb.
        INT32_MIN = never, INT32_MAX = always."""
        ka = np.zeros(self.T, np.int32)
        kb = np.zeros(self.T, np.int32)
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(_lib.lib().sgmm_bundle_thresholds(self.handle, _ptr(ka), _ptr(kb), st))
        return ka, kb

    def close(self):
        if getattr(self, "_h", None):
            h, self._h = self._h, C.c_void_p()
            _lib.release("sgmm_bundle_destroy", h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return self.T


def bundle_windows(askprice1, bidprice1, p_buy_max, p_sell_min, event_step, n_signals, device=None):
    """The per-day window loop of ``load_signals_bundle`` (pipeline/agent_trainer.py:47-73) on the device:
    returns ``(mid_next, best_ask, best_bid, buy_max, sell_min)``, ``n_signals - 1`` float64 values each."""
    if device is None:
        device = torch.cuda.current_device()
    cols = [np.ascontiguousarray(a, np.float64) for a in (askprice1, bidprice1, p_buy_max, p_sell_min)]
    E = cols[0].size
    if any(c.ndim != 1 or c.size != E for c in cols):
        raise ValueError("event columns must be 1-D and of equal length")
    m = max(int(n_signals) - 1, 0)
    out = [np.empty(m, np.float64) for _ in range(5)]
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    _lib.check(_lib.lib().sgmm_bundle_windows_host(E, *[_ptr(c) for c in cols], int(event_step), int(n_signals),
                                                   *[_ptr(o) for o in out], int(device), st))
    return tuple(out)


def day_bundle(event_df, s1_pred, s2_pred, event_step=19, device=None):
    """One day of ``load_signals_bundle``: ``event_df`` is anything with the columns askprice1, bidprice1,
    p_buy_max, p_sell_min (a DataFrame or a dict of arrays); returns that day's 7-tuple
    ``(s1, s2, mid_next, best_ask, best_bid, buy_max, sell_min)`` (agent_trainer.py:47-73)."""
    s1_pred, s2_pred = np.asarray(s1_pred), np.asarray(s2_pred).reshape(-1)
    n = min(len(s1_pred), len(s2_pred))                                    # :47
    col = (lambda k: np.asarray(event_df[k]))
    mid, ask, bid, bmax, smin = bundle_windows(col("askprice1"), col("bidprice1"), col("p_buy_max"), col("p_sell_min"),
                                               event_step, n, device)
    return s1_pred[-n:][:-1] if n else s1_pred[:0], s2_pred[-n:][:-1] if n else s2_pred[:0], mid, ask, bid, bmax, smin


def concat_days(days):
    """``np.concatenate`` of per-day 7-tuples (agent_trainer.py:75-77): a multi-day bundle is ONE episode."""
    return tuple(np.concatenate([d[k] for d in days]) for k in range(7))
