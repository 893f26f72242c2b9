// sgmm_prep.cu -- the steps immediately upstream and downstream of the rollout (SURVEY.md 8f rows 3 and 4):
//
//   bundle_windows_kernel   the per-day window loop of load_signals_bundle (pipeline/agent_trainer.py:47-73):
//                           event sampling every `step` events, NaN-skipping max / min of p_buy_max /
//                           p_sell_min over each inclusive window, ask / bid gather at the current sample,
//                           mid of the next sample.  One thread per output bar; HBM-bound:
//                           (step+1) * 16 B + 32 B read, 40 B written per bar.
//   analytics_kernel        StrategyAnalytics.summary_dict (analytics/mm_analyzer.py:5-56) for a batch of
//                           traces: total PnL, MAP, PnL/MAP, max drawdown, trade Sharpe, trade count.
//                           pandas reduces float64 with numpy's pairwise summation; the kernel follows the
//                           same association (8-way blocks of <= 128, halves rounded to a multiple of 8) so the
//                           Sharpe ratio is bit-identical to the reference's.  One warp per trace: lanes stream
//                           the trace through shared memory, lane 0 runs the order-sensitive recurrences.
#include <cmath>
#include "sgmm_internal.h"
#include "sgmm_step_core.h"
#include "sgmm_np_sum.cuh"

namespace sgmm {

__global__ void bundle_windows_kernel(int64_t E, const double* __restrict__ ask1, const double* __restrict__ bid1,
                                      const double* __restrict__ pmax, const double* __restrict__ pmin,
                                      int64_t step, int64_t k0, int64_t nbars,
                                      double* __restrict__ mid_next, double* __restrict__ best_ask, double* __restrict__ best_bid,
                                      double* __restrict__ buy_max, double* __restrict__ sell_min)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nbars) return;
    const int64_t a = (k0 + i) * step, b = a + step;                      // agent_trainer.py:55-57 (inclusive window)
    double mx = NAN, mn = NAN;
    for (int64_t e = a; e <= b; ++e) {
        const double x = pmax[e], y = pmin[e];
        if (x == x && !(mx >= x)) mx = x;                                 // :58  pandas max skips NaN; NaN if none
        if (y == y && !(mn <= y)) mn = y;                                 // :59
    }
    buy_max[i] = mx; sell_min[i] = mn;
    best_ask[i] = ask1[a]; best_bid[i] = bid1[a];                         // :70-71 current sample
    mid_next[i] = __ddiv_rn(add_rn(ask1[b], bid1[b]), 2.0);               // :73    next sample
}

int launch_bundle_windows(int64_t E, const double* ask1, const double* bid1, const double* pmax, const double* pmin,
                          int64_t step, int64_t n, double* mid_next, double* best_ask, double* best_bid,
                          double* buy_max, double* sell_min, cudaStream_t st)
{
    if (E < 0 || step <= 0 || n < 0) { set_error("negative size / non-positive step"); return SGMM_ERR_INVALID; }
    if (n <= 1 || E == 0) return SGMM_OK;
    const int64_t S = (E + step - 1) / step;
    if (n > S) { set_error("%lld signals but only %lld sampled events (ceil(%lld / %lld))", (long long)n, (long long)S, (long long)E, (long long)step); return SGMM_ERR_INVALID; }
    const int64_t nbars = n - 1;
    bundle_windows_kernel<<<(unsigned)((nbars + 127) / 128), 128, 0, st>>>(E, ask1, bid1, pmax, pmin, step, S - n, nbars,
                                                                           mid_next, best_ask, best_bid, buy_max, sell_min);
    return check_cuda(cudaGetLastError(), "bundle_windows_kernel launch");
}

// One warp per trace.  wealth == nullptr: wealth[t] = cash[t] + inventory[t] * mid[t]  (Env/recorder.py:46).
__global__ void analytics_kernel(int64_t B, int64_t T, const double* __restrict__ wealth, const double* __restrict__ cash,
                                 const double* __restrict__ mid, const int32_t* __restrict__ inventory,
                                 const uint8_t* __restrict__ is_trade, double* __restrict__ scratch, double* __restrict__ out)
{
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (b >= B) return;
    const int32_t* iv = inventory + b * T;
    const uint8_t* tr = is_trade + b * T;
    double* sc = scratch + b * T;
    double* o = out + b * 6;
    if (T <= 0) { if (lane < 6) o[lane] = 0.0; return; }
    auto wealth_at = [&](int64_t t) -> double {
        return wealth ? wealth[b * T + t] : add_rn(cash[b * T + t], mul_rn((double)iv[t], mid[t]));
    };
    // pass 1 (all lanes): |inventory| sum, trade count, and the wealth column materialised into scratch
    long long abs_sum = 0; int trades = 0;
    for (int64_t t = lane; t < T; t += 32) {
        const int32_t v = iv[t];
        abs_sum += v < 0 ? -(long long)v : v;
        trades += tr[t] ? 1 : 0;
        sc[t] = wealth_at(t);
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        abs_sum += __shfl_xor_sync(0xffffffffu, abs_sum, off);
        trades += __shfl_xor_sync(0xffffffffu, trades, off);
    }
    __syncwarp();
    if (lane != 0) return;
    // pass 2 (lane 0): the order-sensitive part -- running maximum, drawdown, wealth differences of trade rows
    const double w0 = sc[0], wl = sc[T - 1];
    double cmax = w0, dd = 0.0, prev = 0.0;
    int64_t m = 0; bool seen = false;
    for (int64_t t = 0; t < T; ++t) {
        const double w = sc[t];
        if (w > cmax) cmax = w;                                        // mm_analyzer.py:20
        const double d = sub_rn(w, cmax);                              // :21
        if (t == 0 || d < dd) dd = d;                                  // :22
        if (tr[t]) {                                                   // :10, :39  (in place: m <= t)
            if (seen) sc[m++] = sub_rn(w, prev);
            prev = w; seen = true;
        }
    }
    const double total = sub_rn(wl, w0);                               // :15
    const double map = __ddiv_rn((double)abs_sum, (double)T);          // :27
    const double sharpe = trade_sharpe(sc, m, trades);                  // :36-45, pandas mean / std(ddof=1)
    o[0] = total; o[1] = map; o[2] = map == 0.0 ? 0.0 : __ddiv_rn(total, map); o[3] = dd; o[4] = sharpe; o[5] = (double)trades;
}

int launch_analytics(int64_t B, int64_t T, const double* wealth, const double* cash, const double* mid,
                     const int32_t* inventory, const uint8_t* is_trade, double* scratch, double* out, cudaStream_t st)
{
    if (B < 0 || T < 0) { set_error("negative size"); return SGMM_ERR_INVALID; }
    if (B == 0) return SGMM_OK;
    if (!inventory || !is_trade || !scratch || !out || (!wealth && (!cash || !mid))) { set_error("NULL array"); return SGMM_ERR_INVALID; }
    const int warps = 4;
    analytics_kernel<<<(unsigned)((B + warps - 1) / warps), warps * 32, 0, st>>>(B, T, wealth, cash, mid, inventory, is_trade, scratch, out);
    return check_cuda(cudaGetLastError(), "analytics_kernel launch");
}

}  // namespace sgmm
