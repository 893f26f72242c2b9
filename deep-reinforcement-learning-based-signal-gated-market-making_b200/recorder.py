"""StrategyRecorder with the reference's row contract (Env/recorder.py:4-52), plus a constructor
from the device trace so that a whole blind test / backtest is ONE kernel launch instead of a
per-bar Python loop (pipeline/agent_trainer.py:144-153, main.py:63-90).
"""
from __future__ import annotations

import numpy as np

_LIST_COLUMNS = ['step', 'mid', 'ask', 'bid', 'off_a', 'off_b', 'reward', 'inventory', 'cash',
                 'pnl_reward', 'inventory_reward', 'fee_paid', 'is_trade']


class StrategyRecorder:
    def __init__(self):
        self.data = []

    # -- the reference's two per-step entry points (recorder.py:8-36) -----------------------------
    def record(self, step, mid, ask, bid, action, reward, inv, cash, info):
        self.data.append([step, mid, ask, bid, action[0], action[1], reward, inv, cash,
                          info['pnl_reward'], info['inventory_reward'], info.get('fee_paid', 0.0),
                          (info['fill_buy'] or info['fill_sell'])])

    def record_detailed(self, step, mid, ask, bid, action, reward, inv, cash, info, s1, s2):
        self.data.append({
            'step': step, 'mid': mid, 'best_ask': ask, 'best_bid': bid,
            'off_a': action[0], 'off_b': action[1], 'reward': reward, 'inventory': inv, 'cash': cash,
            'pnl_reward': info['pnl_reward'], 'inventory_reward': info['inventory_reward'],
            'fee_paid': info.get('fee_paid', 0.0), 'fill_buy': info['fill_buy'],
            'fill_sell': info['fill_sell'], 's1_pred': s1, 's2_pred': s2})

    # -- device trace -> rows (main.py:74-90 layout: ask/bid keys, fills, signals) ----------------
    @classmethod
    def from_trace(cls, trace, bundle):
        """``trace``: dict from :func:`engine.rollout_trace`, or row i of a population trace moved to numpy
        (``{k: v[i].cpu().numpy() for k, v in engine.rollout_trace_population(...)[2].items()}``, all columns);
        ``bundle``: the host 7-tuple."""
        s1, s2, mid, ask, bid = (np.asarray(bundle[i]) for i in range(5))
        rec = cls()
        T = len(mid)
        rec._frame = {
            'step': np.arange(T, dtype=np.int64), 'mid': mid, 'ask': ask, 'bid': bid,
            'off_a': trace['off_a'], 'off_b': trace['off_b'], 'reward': trace['reward'],
            'inventory': trace['inventory'].astype(np.int64), 'cash': trace['cash'],
            'fee_paid': trace['fee_paid'], 's1_pred': s1, 's2_pred': s2,
            'pnl_reward': trace['pnl_reward'], 'inventory_reward': trace['inventory_reward'],
            'fill_buy': trace['fill_buy'].astype(np.int64), 'fill_sell': trace['fill_sell'].astype(np.int64),
        }
        # the derived columns of recorder.py:45-51 come from the same kernel pass (sequential fp64 running sums in bar
        # order == pandas cumsum); to_dataframe only attaches them
        rec._derived = {k: (trace[k].astype(np.int64) if k == 'skew' else trace[k])
                        for k in ('spread', 'wealth', 'cum_reward', 'skew', 'cum_fees', 'unrealized_pnl') if k in trace}
        return rec

    def to_dataframe(self):
        import pandas as pd
        if getattr(self, "_frame", None) is not None:
            df = pd.DataFrame(self._frame)
        elif len(self.data) > 0 and isinstance(self.data[0], list):
            df = pd.DataFrame(self.data, columns=_LIST_COLUMNS)
        else:
            df = pd.DataFrame(self.data)
            # record_detailed writes best_ask/best_bid while the derived columns read ask/bid
            # (recorder.py:22-23 vs :45): expose both names instead of raising KeyError
            if 'ask' not in df.columns and 'best_ask' in df.columns:
                df['ask'] = df['best_ask']
                df['bid'] = df['best_bid']
        d = getattr(self, "_derived", None)
        if d is not None and len(d) == 6:          # device trace: derived columns already computed by the kernel
            df['spread'] = d['spread']; df['wealth'] = d['wealth']; df['cum_reward'] = d['cum_reward']
            df['skew'] = d['skew']; df['cum_fees'] = d['cum_fees']; df['realized_pnl'] = df['cash']
            df['unrealized_pnl'] = d['unrealized_pnl']
            return df
        # derived columns (recorder.py:45-51) for rows recorded one by one on the host
        df['spread'] = df['ask'] - df['bid']
        df['wealth'] = df['cash'] + df['inventory'] * df['mid']
        df['cum_reward'] = df['reward'].cumsum()
        df['skew'] = df['off_b'] - df['off_a']
        df['cum_fees'] = df['fee_paid'].cumsum()
        df['realized_pnl'] = df['cash']
        df['unrealized_pnl'] = df['inventory'] * df['mid']
        return df
