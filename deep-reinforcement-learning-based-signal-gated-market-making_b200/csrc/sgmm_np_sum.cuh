// sgmm_np_sum.cuh -- numpy's pairwise float64 summation on the device, defined once for every kernel that restates a
// pandas / numpy reduction bit for bit: analytics_kernel (sgmm_prep.cu) and the trade-Sharpe objective of
// walk_account_kernel (sgmm_one.cu).
#pragma once
#include <stdint.h>
#include <cmath>
#include "sgmm_step_core.h"

namespace sgmm {

// numpy's pairwise_sum over a[0..n) (float64), same association: blocks of <= 128 elements are summed with
// eight interleaved accumulators, larger ranges are split at (n/2 rounded down to a multiple of 8) and the halves
// added.  The recursion is run on an explicit stack (depth <= log2(n/128) + 1) so the frame size is static.
__device__ __forceinline__ double np_block_sum(const double* a, int64_t n)
{
    if (n < 8) {
        double res = 0.0;
        for (int64_t i = 0; i < n; ++i) res = add_rn(res, a[i]);
        return res;
    }
    double r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = a[k];
    int64_t i;
    for (i = 8; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = add_rn(r[k], a[i + k]);
    }
    double res = add_rn(add_rn(add_rn(r[0], r[1]), add_rn(r[2], r[3])), add_rn(add_rn(r[4], r[5]), add_rn(r[6], r[7])));
    for (; i < n; ++i) res = add_rn(res, a[i]);
    return res;
}

static __device__ double np_pairwise_sum(const double* a, int64_t n)
{
    struct Frame { int64_t off, n; double left; int stage; };
    Frame st[48];
    int sp = 0;
    st[0].off = 0; st[0].n = n; st[0].left = 0.0; st[0].stage = 0;
    double ret = 0.0;
    while (sp >= 0) {
        Frame& f = st[sp];
        if (f.stage == 0) {
            if (f.n <= 128) { ret = np_block_sum(a + f.off, f.n); --sp; }
            else {
                int64_t n2 = f.n / 2; n2 -= n2 % 8;
                f.stage = 1;
                st[sp + 1].off = f.off; st[sp + 1].n = n2; st[sp + 1].stage = 0;
                ++sp;
                continue;
            }
        } else if (f.stage == 1) {                     // left half returned
            int64_t n2 = f.n / 2; n2 -= n2 % 8;
            f.left = ret; f.stage = 2;
            st[sp + 1].off = f.off + n2; st[sp + 1].n = f.n - n2; st[sp + 1].stage = 0;
            ++sp;
            continue;
        } else {                                       // right half returned
            ret = add_rn(f.left, ret); --sp;
        }
    }
    return ret;
}

// The trade Sharpe ratio of StrategyAnalytics (analytics/mm_analyzer.py:36-45: pandas mean / std with ddof = 1) over the
// m = trades - 1 wealth differences d[0..m) of consecutive trade rows: 0 below two trades, NaN for a single difference,
// 0 when the std is 0.  d is overwritten by the squared deviations.
__device__ __forceinline__ double trade_sharpe(double* d, int64_t m, int trades)
{
    double sharpe = 0.0;
    if (trades >= 2) {
        const double mean = __ddiv_rn(np_pairwise_sum(d, m), (double)m);
        for (int64_t i = 0; i < m; ++i) { const double x = sub_rn(mean, d[i]); d[i] = mul_rn(x, x); }
        const double var = m > 1 ? __ddiv_rn(np_pairwise_sum(d, m), (double)(m - 1)) : NAN;
        const double sd = __dsqrt_rn(var);
        sharpe = sd != sd ? NAN : (sd == 0.0 ? 0.0 : __ddiv_rn(mean, sd));
    }
    return sharpe;
}

}  // namespace sgmm
