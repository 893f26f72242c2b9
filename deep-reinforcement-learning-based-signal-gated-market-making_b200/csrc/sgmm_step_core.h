// sgmm_step_core.h -- one MDP step of the First-Passage-Time env, host + device.
//
// Restates /root/reference/Env/market_env.py:22-67 with every fp64 operation written as an
// explicitly un-fused IEEE-754 op (__dmul_rn / __dadd_rn on the device; the host TU is compiled
// with -ffp-contract=off), because the reference evaluates `best + off*tick` as two roundings and
// ~10 % of exact-touch cases flip if the product is fused (SURVEY.md 7.4-2).
#pragma once
#include <stdint.h>
#include "../../include/sgmm.h"

#if defined(__CUDACC__)
#define SGMM_HD __host__ __device__ __forceinline__
#else
#define SGMM_HD static inline
#endif

namespace sgmm {

SGMM_HD double mul_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    volatile double r = a * b; return r;
#endif
}
SGMM_HD double add_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    volatile double r = a + b; return r;
#endif
}
SGMM_HD double sub_rn(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, -b);          // a - b == a + (-b) exactly in IEEE-754
#else
    volatile double r = a - b; return r;
#endif
}

// market_env.py:30-31.  Offsets are ticks: integers from the policies (drl_engine.py:39), but the env itself takes
// whatever the caller passes (:23) -- an unrounded benchmark offset such as 1.7 quotes at 1.7 ticks -- hence the
// double overloads (int -> double is exact for |off| < 2^53, so both give the same quote for integral offsets).
SGMM_HD double quote_ask(double best_ask, double off_a, double tick) { return add_rn(best_ask, mul_rn(off_a, tick)); }
SGMM_HD double quote_bid(double best_bid, double off_b, double tick) { return sub_rn(best_bid, mul_rn(off_b, tick)); }
SGMM_HD double quote_ask(double best_ask, int64_t off_a, double tick) { return quote_ask(best_ask, (double)off_a, tick); }
SGMM_HD double quote_bid(double best_bid, int64_t off_b, double tick) { return quote_bid(best_bid, (double)off_b, tick); }
SGMM_HD double quote_ask(double best_ask, int off_a, double tick) { return quote_ask(best_ask, (double)off_a, tick); }
SGMM_HD double quote_bid(double best_bid, int off_b, double tick) { return quote_bid(best_bid, (double)off_b, tick); }

// market_env.py:46,48 and :52,54 -- the P&L leg of one filled side at its quoted price, fee term included.  FEE = false
// drops the fee term, for callers that have checked fee_rate == 0.
template <bool FEE = true>
SGMM_HD double buy_leg(double my_bid, double mid_next, double fee_rate)
{
    const double leg = sub_rn(mid_next, my_bid);
    return FEE ? sub_rn(leg, mul_rn(my_bid, fee_rate)) : leg;
}
template <bool FEE = true>
SGMM_HD double sell_leg(double my_ask, double mid_next, double fee_rate)
{
    const double leg = sub_rn(my_ask, mid_next);
    return FEE ? sub_rn(leg, mul_rn(my_ask, fee_rate)) : leg;
}

// market_env.py:57 -- phi * |inventory| for the three values |inventory| takes in the reference's env (i_max = -i_min = 2)
struct PenaltyTable { double p0, p1, p2; };
SGMM_HD PenaltyTable penalty_table(double phi) { return {mul_rn(phi, 0.0), mul_rn(phi, 1.0), mul_rn(phi, 2.0)}; }
// (The copies make the select one over values, which keeps the branch layout the hot loops were tuned with; nvcc lays out
// a select over struct members differently.)
SGMM_HD double penalty(const PenaltyTable& pen, int abs_inventory)
{
    const double p0 = pen.p0, p1 = pen.p1, p2 = pen.p2;
    return abs_inventory == 0 ? p0 : (abs_inventory == 1 ? p1 : p2);
}

// drl_engine.py:64-65 -- an episode without a single trade loses 50
SGMM_HD double episode_fitness(double total, int trades) { return trades == 0 ? sub_rn(total, 50.0) : total; }
// the fitness of a StrategyAnalytics objective value v (sgmm.h, SGMM_OBJECTIVE_*): the same -50 without trades, and a NaN
// objective (the Sharpe of exactly two trades) is -50 too, since the GA's ranking would put it first
SGMM_HD double objective_fitness(double v, int trades) { return trades == 0 ? sub_rn(v, 50.0) : (v != v ? -50.0 : v); }

// market_env.py:22-67.  off_a/off_b already include the adversary's displacement (:25-28).  Off = int64_t or double.
template <typename Off>
SGMM_HD void env_step(sgmm_env_state& e, Off off_a, Off off_b,
                      double mid_next, double best_ask, double best_bid,
                      double buy_max, double sell_min, sgmm_step_info& out)
{
    const double my_ask = quote_ask(best_ask, off_a, e.tick_size);
    const double my_bid = quote_bid(best_bid, off_b, e.tick_size);
    const bool can_buy = e.inventory < e.i_max;                    // :34  (pre-step inventory)
    const bool can_sell = e.inventory > e.i_min;                   // :35
    const bool fill_buy = can_buy && (my_bid >= sell_min);         // :37  NaN -> false
    const bool fill_sell = can_sell && (my_ask <= buy_max);        // :38
    double pnl = 0.0, fee_paid = 0.0;
    if (fill_buy) {                                                // :44-49
        e.inventory += 1;
        const double fee = mul_rn(my_bid, e.fee_rate);
        e.cash = sub_rn(e.cash, add_rn(my_bid, fee));
        pnl = add_rn(pnl, buy_leg(my_bid, mid_next, e.fee_rate));
        fee_paid = add_rn(fee_paid, fee);
    }
    if (fill_sell) {                                               // :50-55
        e.inventory -= 1;
        const double fee = mul_rn(my_ask, e.fee_rate);
        e.cash = add_rn(e.cash, sub_rn(my_ask, fee));
        pnl = add_rn(pnl, sell_leg(my_ask, mid_next, e.fee_rate));
        fee_paid = add_rn(fee_paid, fee);
    }
    const int64_t ai = e.inventory < 0 ? -e.inventory : e.inventory;
    const double pen = mul_rn(e.phi, (double)ai);                  // :57
    out.reward = sub_rn(pnl, pen);                                 // :58
    out.pnl_reward = pnl;
    out.inventory_reward = -pen;
    out.fee_paid = fee_paid;
    out.fill_buy = fill_buy ? 1 : 0;
    out.fill_sell = fill_sell ? 1 : 0;
}

}  // namespace sgmm
