// sgmm_rollout.cu -- population rollout of the signal-gated market-making MDP on sm_100a.
//
// One episode per individual = /root/reference/Env/drl_engine.py:9-67 (evaluate_individual):
//   state build (:33-35) -> TradingPolicy.forward (models/model.py:9-15) -> x5 + round-half-even
//   (:39) -> optional adversary displacement (:42-48, models/model.py:40-50) -> FTPEnv.step
//   (Env/market_env.py:22-67) -> fp64 reward sum (:54) -> trade count (:60-61) -> -50 penalty (:64).
//
// Mapping (see DESIGN.md section 4):
//   * a warp owns U individuals (U = 1, 2 or 4); each individual is spread over L = 32/U lanes and
//     every lane keeps U rows of W2 (+ its slices of W1/b1/b2/W3) in REGISTERS for the whole
//     episode -- the per-individual GEMV has no batch dimension, so weights-in-registers with the
//     activations broadcast through shared memory is the shape that keeps the FP32 pipe fed;
//   * the hidden layer runs as packed fma.rn.f32x2 (FFMA2, new on sm_100): the two halves are two
//     of the four interleaved accumulation chains of the SGMM-F32 order;
//   * the 32->2 output layer is a butterfly of warp shuffles;
//   * bars are shared by the whole population: a 4-stage ring of 128-bar chunks is streamed
//     L2 -> shared memory with cp.async.bulk (TMA 1-D bulk copies) completing on mbarriers; warps
//     release a stage through an "empty" mbarrier and a dedicated producer warp refills it;
//   * the env step is branch-free: fills are integer compares against per-bar thresholds derived
//     once per bundle with the reference's exact fp64 expression, inventory is an integer;
//   * quotes / P&L / penalty / reward sum -- un-fused fp64 in the reference's order -- are NOT in the
//     step loop: the compute warps hand one 8-byte record per bar through shared memory to the CTA's
//     producer warp, whose lane j accounts individual j of the CTA (one fp64 warp instruction for all 28
//     individuals instead of one per compute warp, and no int -> fp64 conversions or fp64 registers in the
//     step loop).  Measured at P = 4096 x 14 400 bars: 5.25 ms with the accounting in the loop, 4.53 ms this way.
#include <cstdio>
#include <cstdlib>
#include "sgmm_internal.h"
#include "sgmm_rng.cuh"
#include "sgmm_adversary.cuh"
#include "sgmm_step_core.h"

namespace sgmm {

constexpr int RING_STAGES = 4;
constexpr int CHUNK_BARS = 128;
constexpr int MAX_WARPS = 16;
constexpr int REC_STAGES = 2;             // chunks of step records in flight between the compute warps and the accounting warp

// ---------------------------------------------------------------------------------------------
// mbarrier / TMA bulk-copy helpers (raw PTX)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE_%=;\n"
        "bra LAB_WAIT_%=;\n"
        "LAB_DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---------------------------------------------------------------------------------------------
// bundle prologue: pack bars and derive the integer fill thresholds
// ---------------------------------------------------------------------------------------------
template <bool ASK>
__device__ __forceinline__ bool touch(double best, int k, double tick, double bound)
{
    // market_env.py:30-31,37-38 -- the exact two-rounding quote and the exact comparison
    return ASK ? (quote_ask(best, k, tick) <= bound) : (quote_bid(best, k, tick) >= bound);
}

template <bool ASK>
__device__ int32_t fill_threshold_plus1(double best, double tick, double bound)
{
    // the quote is monotone in k (IEEE rounding is monotone), so {k : touch} is a down-set
    if (!touch<ASK>(best, -K_CLAMP, tick, bound)) return K_NEVER;     // includes NaN bounds
    if (touch<ASK>(best, K_CLAMP, tick, bound)) return K_ALWAYS;
    // touch(lo) true, touch(hi) false; 64-bit because hi - lo spans 2^31 before the search narrows it
    int64_t lo = -K_CLAMP, hi = K_CLAMP;
    // warm start: the real-arithmetic solution is within a few ticks of the answer
    const double est = ASK ? (bound - best) / tick : (best - bound) / tick;
    if (est > -1.0e9 && est < 1.0e9) {
        const int e = (int)floor(est);
        if (e - 4 > lo && touch<ASK>(best, e - 4, tick, bound)) lo = e - 4;
        if (e + 4 < hi && !touch<ASK>(best, e + 4, tick, bound)) hi = e + 4;
    }
    while (hi - lo > 1) {
        const int64_t mid = lo + (hi - lo) / 2;
        if (touch<ASK>(best, (int)mid, tick, bound)) lo = mid; else hi = mid;
    }
    return (int32_t)(lo + 1);
}

// fill <=> rint_half_even(q) <= K  <=>  q < K + 0.5, or q == K + 0.5 exactly and K is even (the tie
// rounds down to K).  Folding the tie into a strict compare: threshold = K + 0.5, moved one ulp up
// when K is even -- for -2^23 <= K < 2^23, where K + 0.5 is exact in fp32.  Beyond, the q that can
// round to the far side of K are fp32 numbers of magnitude >= 2^23, all integers: fill <=> q <= K
// <=> q < the next float above the largest float <= K.  Exact for every threshold the prologue
// derives (|K| <= K_CLAMP).
__device__ __forceinline__ float float_threshold(int32_t k_plus1)
{
    if (k_plus1 == K_NEVER) return -INFINITY;
    if (k_plus1 == K_ALWAYS) return INFINITY;
    const int32_t K = k_plus1 - 1;
    if (K < -(1 << 23) || K >= (1 << 23)) return nextafterf(__int2float_rd(K), INFINITY);
    const float t = (float)K + 0.5f;                  // exact
    return (K & 1) == 0 ? nextafterf(t, INFINITY) : t;
}

__global__ void bundle_prologue_kernel(int64_t T, const float* __restrict__ z1, const float* __restrict__ z2,
                                       const double* __restrict__ mid, const double* __restrict__ ask,
                                       const double* __restrict__ bid, const double* __restrict__ bmax,
                                       const double* __restrict__ smin, double tick,
                                       BarSig* __restrict__ sig, BarPx* __restrict__ px)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    BarSig s;
    s.z1 = z1[t]; s.z2 = z2[t];
    s.ka1 = fill_threshold_plus1<true>(ask[t], tick, bmax[t]);
    s.kb1 = fill_threshold_plus1<false>(bid[t], tick, smin[t]);
    s.tha = float_threshold(s.ka1);
    s.thb = float_threshold(s.kb1);
    s.pad0 = s.pad1 = 0;
    sig[t] = s;
    BarPx p; p.ask = ask[t]; p.bid = bid[t]; p.mid_next = mid[t]; p.pad = 0.0;
    px[t] = p;
}

int launch_prologue(sgmm_bundle* b, const float* z1, const float* z2, const double* mid,
                    const double* ask, const double* bid, cudaStream_t st)
{
    if (b->T == 0) return SGMM_OK;
    const int threads = 128;
    const int64_t blocks = (b->T + threads - 1) / threads;
    bundle_prologue_kernel<<<(unsigned)blocks, threads, 0, st>>>(b->T, z1, z2, mid, ask, bid, b->bmax, b->smin,
                                                                  b->tick, b->sig, b->px);
    return check_cuda(cudaGetLastError(), "bundle_prologue_kernel launch");
}

// ---------------------------------------------------------------------------------------------
// the rollout kernel (H = 32)
// ---------------------------------------------------------------------------------------------
// compute warps per CTA (one more warp is the producer): bounded by the register file
__host__ __device__ constexpr int max_compute_warps(int U) { return U == 4 ? 7 : (U == 2 ? 15 : MAX_WARPS); }

struct RingSmem {
    uint64_t full[RING_STAGES];
    uint64_t empty[RING_STAGES];
    BarSig sig[RING_STAGES][CHUNK_BARS];
    BarPx px[RING_STAGES][CHUNK_BARS];   // prices: read by the accounting warp only
    float hbuf[MAX_WARPS][128];          // per warp: U individuals x 32 activations, 16-B interleaved
    float rbuf[MAX_WARPS][80];           // per warp: 4 individuals x 8 lanes x (pa,pb), group stride 20 words
    // step records handed to the accounting warp: one 8-byte code per (bar of the chunk, individual of the CTA)
    uint64_t rec_full[REC_STAGES];
    uint64_t rec_empty[REC_STAGES];
    uint64_t rec[REC_STAGES][CHUNK_BARS][32];
#ifdef SGMM_ROLLOUT_TRACE
    long long trace[2][64][3];
#endif
};

template <int U, bool ADV, bool FEE>
__global__ void __launch_bounds__((max_compute_warps(U) + 1) * 32, 1)
rollout_kernel_h32(const RolloutArgs a)
{
    constexpr int H = 32;
    constexpr int NI = U;                // individuals per warp
    constexpr int L = 32 / U;            // lanes per individual
    constexpr int64_t G = (int64_t)H * H + 7 * H + 2;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    RingSmem& sm = *reinterpret_cast<RingSmem*>(smem_raw);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = (blockDim.x >> 5) - 1;          // compute warps; the last warp is the TMA producer
    const int g = lane / L, l = lane % L;
    const int64_t first = (int64_t)blockIdx.x * nwarps * NI;
    const int64_t remaining = a.mm.count - first;
    const int live_warps = (int)(remaining >= (int64_t)nwarps * NI ? nwarps : (remaining + NI - 1) / NI);
    const int64_t ind = first + (int64_t)warp * NI + g;
    const bool live = ind < a.mm.count;
    const int64_t T = a.T;
    const int64_t nchunks = (T + CHUNK_BARS - 1) / CHUNK_BARS;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < RING_STAGES; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], live_warps); }
#pragma unroll
        for (int r = 0; r < REC_STAGES; ++r) { mbar_init(&sm.rec_full[r], live_warps); mbar_init(&sm.rec_empty[r], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == nwarps) {
        // ===== the CTA's last warp: TMA producer of the bar ring AND the fp64 half of the env step =====
        // The compute warps do the policy and the INTEGER half of the step and hand one 8-byte record per bar and
        // individual through shared memory; here lane j accounts individual first + j: quotes, P&L legs, penalty and
        // the bar-order reward sum in the reference's un-fused fp64 (market_env.py:30-58, drl_engine.py:54).  One
        // warp instruction per fp64 operation for ALL individuals of the CTA -- in the step loop the same arithmetic
        // was issued once per compute warp (22 of 217 instructions, two of them conversions on the XU pipe, plus the
        // fp64 live ranges in a 254-register kernel) and cost 16 % of the loop.
        const int64_t indj = first + lane;
        const bool livej = lane < live_warps * NI && indj < a.mm.count;
        const double tick = a.tick, fee = a.fee;
        const PenaltyTable pen = penalty_table(a.phi);
        double total = 0.0;                                              // drl_engine.py:26
        int ntr = 0, inv = 0;                                            // market_env.py:17
        int64_t next_load = 0;
        for (int64_t c = 0; c < nchunks; ++c) {
            // keep the bar ring RING_STAGES chunks ahead of the chunk being accounted
            const int64_t lim = c + RING_STAGES < nchunks ? c + RING_STAGES : nchunks;
            for (; next_load < lim; ++next_load) {
                if (lane == 0) {
                    const int s = (int)(next_load % RING_STAGES);
                    if (next_load >= RING_STAGES) mbar_wait(&sm.empty[s], (uint32_t)(((next_load / RING_STAGES) - 1) & 1));
                    const int64_t tl = next_load * CHUNK_BARS;
                    const uint32_t nb = (uint32_t)(T - tl < CHUNK_BARS ? T - tl : CHUNK_BARS);
                    mbar_arrive_expect_tx(&sm.full[s], nb * (uint32_t)(sizeof(BarSig) + sizeof(BarPx)));
                    tma_bulk_g2s(&sm.sig[s][0], a.sig + tl, nb * (uint32_t)sizeof(BarSig), &sm.full[s]);
                    tma_bulk_g2s(&sm.px[s][0], a.px + tl, nb * (uint32_t)sizeof(BarPx), &sm.full[s]);
                }
            }
            __syncwarp();
            const int r = (int)(c % REC_STAGES);
            mbar_wait(&sm.rec_full[r], (uint32_t)((c / REC_STAGES) & 1));
            const int64_t t0 = c * CHUNK_BARS;
            const int n = (int)(T - t0 < CHUNK_BARS ? T - t0 : CHUNK_BARS);
            // the chunk's prices sit in its ring stage (complete: the compute warps waited for the same barrier, and
            // the stage is refilled by this warp only after this loop)
            const BarPx* pxs = &sm.px[c % RING_STAGES][0];
#pragma unroll 4
            for (int i = 0; i < n; ++i) {
                const uint64_t code = sm.rec[r][i][lane];
                int ka = (int)(uint32_t)code, kb = (int)(uint32_t)(code >> 32);
                const bool fs = ka != (ADV ? SGMM_CODE_NOFILL : SGMM_CODE_NOFILL_F), fb = kb != (ADV ? SGMM_CODE_NOFILL : SGMM_CODE_NOFILL_F);
                inv += (fb ? 1 : 0) - (fs ? 1 : 0);                      // market_env.py:45,51
                const int ai = inv < 0 ? -inv : inv;
                const bool traded = fb || fs;
                ntr += traded ? 1 : 0;                                   // drl_engine.py:60-61
                double pnl = 0.0;                                        // market_env.py:40
                if (__any_sync(0xffffffffu, traded)) {
                    const double2 ab = *reinterpret_cast<const double2*>(&pxs[i].ask);
                    const double mid = pxs[i].mid_next;
                    if (!ADV) { ka = __float2int_rn(__int_as_float(ka)); kb = __float2int_rn(__int_as_float(kb)); }   // drl_engine.py:39
                    const double my_ask = quote_ask(ab.x, ka, tick), my_bid = quote_bid(ab.y, kb, tick);      // market_env.py:30-31
                    const double leg_b = buy_leg<FEE>(my_bid, mid, fee), leg_s = sell_leg<FEE>(my_ask, mid, fee);
                    pnl = fb ? add_rn(pnl, leg_b) : pnl;
                    pnl = fs ? add_rn(pnl, leg_s) : pnl;
                }
                total = add_rn(total, sub_rn(pnl, penalty(pen, ai)));                   // market_env.py:58, drl_engine.py:54
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.rec_empty[r]);
        }
        if (livej) { a.fitness[indj] = episode_fitness(total, ntr); a.trades[indj] = ntr; }
        return;
    }
    if (warp >= live_warps) return;

    // ---- weights into registers (models/model.py:31-36 layout) ---------------------------------
    const PopArgs mmp = resolve(a.mm);
    const GenomeSource src = make_source(mmp, live ? ind : 0, G);
    float w1x[U], w1y[U], w1i[U], b1[U], b2[U], w3a[U], w3b[U];
    float2 w2[U][16];
    float b3a = 0.0f, b3b = 0.0f;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int j = l + L * u;
        if (live) {
            w1x[u] = src.at(3 * j + 0); w1y[u] = src.at(3 * j + 1); w1i[u] = src.at(3 * j + 2);
            b1[u] = src.at(3 * H + j);
            b2[u] = src.at(4 * H + H * H + j);
            w3a[u] = src.at(5 * H + H * H + j);
            w3b[u] = src.at(6 * H + H * H + j);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float v[4]; src.at4(4 * H + (int64_t)j * H + 4 * c, v);
                w2[u][2 * c] = make_float2(v[0], v[1]);
                w2[u][2 * c + 1] = make_float2(v[2], v[3]);
            }
        } else {
            w1x[u] = w1y[u] = w1i[u] = b1[u] = b2[u] = w3a[u] = w3b[u] = 0.0f;
#pragma unroll
            for (int c = 0; c < 16; ++c) w2[u][c] = make_float2(0.0f, 0.0f);
        }
    }
    if (live) { b3a = src.at(7 * H + H * H); b3b = src.at(7 * H + H * H + 1); }

    uint32_t adv_t0 = 0x55555555u, adv_t1 = 0x55555555u, adv_t2 = 0x55555555u;   // all (0,0)
    if (ADV) {
        const PopArgs advp = resolve(a.adv);
        const GenomeSource asrc = make_source(advp, live ? ind : 0, (int64_t)1250);
        // the L lanes of an individual split the 20 states, then gather the whole table
        uint32_t mine[3] = {0u, 0u, 0u};
        for (int s = l; s < 20; s += L) {
            const uint32_t e = live ? adversary_entry(asrc, s) : 5u;
            mine[s >> 3] |= e << ((s & 7) * 4);
        }
#pragma unroll
        for (int m = L / 2; m >= 1; m >>= 1) {
#pragma unroll
            for (int k = 0; k < 3; ++k) mine[k] |= __shfl_xor_sync(0xffffffffu, mine[k], m);
        }
        adv_t0 = mine[0]; adv_t1 = mine[1]; adv_t2 = mine[2];
    }

    float* hb = &sm.hbuf[warp][0];
    float* rbw = &sm.rbuf[warp][0];
    int inv = 0, fbp = 0, fsp = 0;
    float inv2 = 0.0f;                                               // inventory / 2.0 (drl_engine.py:35), exact

    // The step loop does the INTEGER half of the env step (offsets, fills, inventory) and hands one 8-byte record per
    // bar to the accounting warp (above): the offset of each side that filled, or a no-fill marker.  Without the
    // adversary the offsets travel as the fp32 q = raw*5 they are rounded from (no conversion in this loop).
    const int slotj = warp * NI + g;                                 // this individual's lane in the accounting warp

    // Two compute warps share a scheduler (warps w and w + 4).  Measured (profiles/r2_exact_phase_trace_*.log, a clock64 trace of
    // both from the SGMM_ROLLOUT_TRACE build): their steps lock at a relative phase of 0.19 whatever the start offset, and
    // forcing strict alternation of the layer-2 bursts with named barriers is SLOWER (4.88 vs 4.66 ms): the FMA pipe's time
    // per pair of warp-steps (2 x ~200 cycles, FFMA2 with three register operands issues every 2.34 cycles) is conserved
    // whatever the interleaving; both experiments were removed again.
    for (int64_t c = 0; c < nchunks; ++c) {
        const int s = (int)(c % RING_STAGES);
        mbar_wait(&sm.full[s], (uint32_t)((c / RING_STAGES) & 1));
        const int r = (int)(c % REC_STAGES);
        if (c >= REC_STAGES) mbar_wait(&sm.rec_empty[r], (uint32_t)(((c / REC_STAGES) - 1) & 1));   // records of chunk c - 2 accounted
        __syncwarp();
        uint64_t* const recs = &sm.rec[r][0][slotj];
        const int64_t t0 = c * CHUNK_BARS;
        const int n = (int)(T - t0 < CHUNK_BARS ? T - t0 : CHUNK_BARS);
        const BarSig* sigs = &sm.sig[s][0];

        // bar 0 of the chunk: signals, thresholds and the inventory-independent part of layer 1
        float4 sg = *reinterpret_cast<const float4*>(&sigs[0]);                     // z1, z2, tha, thb
        int2 kth = *reinterpret_cast<const int2*>(&sigs[0].ka1);
        float A1[U];
#pragma unroll
        for (int u = 0; u < U; ++u) A1[u] = __fmaf_rn(w1y[u], sg.y, __fmaf_rn(w1x[u], sg.x, b1[u]));

#ifdef SGMM_ROLLOUT_TRACE
        const bool trc = blockIdx.x == 0 && (warp & 3) == 0 && lane == 0 && c == 4;
#endif
#pragma unroll 1
        for (int i = 0; i < n; ++i) {
#ifdef SGMM_ROLLOUT_TRACE
            if (trc && i < 64) { long long t; asm volatile("mov.u64 %0, %%clock64; // %1" : "=l"(t) : "f"(inv2)); sm.trace[warp >> 2][i][0] = t; }
#endif
            // ---- layer 1 (inventory term) + ReLU, publish h1 ------------------------------------
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int j = l + L * u;
                hb[((j >> 2) * NI + g) * 4 + (j & 3)] = fmaxf(__fmaf_rn(w1i[u], inv2, A1[u]), 0.0f);
            }
            __syncwarp();
            const float tha = sg.z, thb = sg.w;
            const int ka1 = kth.x, kb1 = kth.y;
            // ---- prefetch bar i+1 and its layer-1 partial (off the critical path) --------------
            const int inext = i + 1 < CHUNK_BARS ? i + 1 : CHUNK_BARS - 1;
            sg = *reinterpret_cast<const float4*>(&sigs[inext]);
            if (ADV) kth = *reinterpret_cast<const int2*>(&sigs[inext].ka1);
            float A1n[U];
#pragma unroll
            for (int u = 0; u < U; ++u) A1n[u] = __fmaf_rn(w1y[u], sg.y, __fmaf_rn(w1x[u], sg.x, b1[u]));
            // ---- layer 2: U rows x 32, packed FFMA2, four chains per row -----------------------
            float2 P[U], Q[U];
#pragma unroll
            for (int u = 0; u < U; ++u) { P[u] = make_float2(b2[u], 0.0f); Q[u] = make_float2(0.0f, 0.0f); }
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const float4 h4 = *reinterpret_cast<const float4*>(&hb[(k * NI + g) * 4]);
                const float2 hlo = make_float2(h4.x, h4.y), hhi = make_float2(h4.z, h4.w);
#pragma unroll
                for (int u = 0; u < U; ++u) {
#ifdef SGMM_ROLLOUT_SCALAR_FMA       // A/B switch: 128 scalar FFMA instead of 64 FFMA2 -- 4.74 instead of 4.51 ms at P = 4096 (same results)
                    P[u].x = __fmaf_rn(w2[u][2 * k].x, hlo.x, P[u].x); P[u].y = __fmaf_rn(w2[u][2 * k].y, hlo.y, P[u].y);
                    Q[u].x = __fmaf_rn(w2[u][2 * k + 1].x, hhi.x, Q[u].x); Q[u].y = __fmaf_rn(w2[u][2 * k + 1].y, hhi.y, Q[u].y);
#else
                    P[u] = __ffma2_rn(w2[u][2 * k], hlo, P[u]);
                    Q[u] = __ffma2_rn(w2[u][2 * k + 1], hhi, Q[u]);
#endif
                }
            }
#ifdef SGMM_ROLLOUT_TRACE
            if (trc && i < 64) { long long t; asm volatile("mov.u64 %0, %%clock64; // %1 %2" : "=l"(t) : "f"(Q[U - 1].y), "f"(P[0].x)); sm.trace[warp >> 2][i][1] = t; }
#endif
            // ---- layer 3: products, local tree, then the cross-lane tree ------------------------
            float pa[U], pb[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const float2 S = __fadd2_rn(P[u], Q[u]);                 // (a0+a2, a1+a3)
                const float h2 = fmaxf(__fadd_rn(S.x, S.y), 0.0f);
                pa[u] = __fmul_rn(w3a[u], h2);
                pb[u] = __fmul_rn(w3b[u], h2);
            }
            float ra, rb;
            if (U == 4) {
                ra = __fadd_rn(__fadd_rn(pa[0], pa[2 % U]), __fadd_rn(pa[1 % U], pa[3 % U]));
                rb = __fadd_rn(__fadd_rn(pb[0], pb[2 % U]), __fadd_rn(pb[1 % U], pb[3 % U]));
                // butterfly over the 8 lanes of the individual, evaluated by every lane from the 8
                // partials exchanged through shared memory (same tree, 1 round trip instead of 3 shuffles)
                *reinterpret_cast<float2*>(&rbw[g * 20 + l * 2]) = make_float2(ra, rb);
                __syncwarp();
                const float4 r01 = *reinterpret_cast<const float4*>(&rbw[g * 20 + 0]);
                const float4 r23 = *reinterpret_cast<const float4*>(&rbw[g * 20 + 4]);
                const float4 r45 = *reinterpret_cast<const float4*>(&rbw[g * 20 + 8]);
                const float4 r67 = *reinterpret_cast<const float4*>(&rbw[g * 20 + 12]);
                const float2 t04 = __fadd2_rn(make_float2(r01.x, r01.y), make_float2(r45.x, r45.y));
                const float2 t15 = __fadd2_rn(make_float2(r01.z, r01.w), make_float2(r45.z, r45.w));
                const float2 t26 = __fadd2_rn(make_float2(r23.x, r23.y), make_float2(r67.x, r67.y));
                const float2 t37 = __fadd2_rn(make_float2(r23.z, r23.w), make_float2(r67.z, r67.w));
                const float2 e = __fadd2_rn(__fadd2_rn(t04, t26), __fadd2_rn(t15, t37));
                ra = e.x; rb = e.y;
            } else {
                if (U == 2) { ra = __fadd_rn(pa[0], pa[1 % U]); rb = __fadd_rn(pb[0], pb[1 % U]); }
                else { ra = pa[0]; rb = pb[0]; }
#pragma unroll
                for (int m = L / 2; m >= 1; m >>= 1) {
                    ra = __fadd_rn(ra, __shfl_xor_sync(0xffffffffu, ra, m));
                    rb = __fadd_rn(rb, __shfl_xor_sync(0xffffffffu, rb, m));
                }
            }
#ifdef SGMM_ROLLOUT_TRACE
            if (trc && i < 64) { long long t; asm volatile("mov.u64 %0, %%clock64; // %1" : "=l"(t) : "f"(ra)); sm.trace[warp >> 2][i][2] = t; }
#endif
            // ---- quantise + fill decision -------------------------------------------------------
            const float qa = __fmul_rn(__fadd_rn(ra, b3a), 5.0f);           // raw*5.0 (drl_engine.py:39)
            const float qb = __fmul_rn(__fadd_rn(rb, b3b), 5.0f);
            int ka = 0, kb = 0;
            bool fb, fs;
            if (ADV) {                                                       // drl_engine.py:42-48
                ka = __float2int_rn(qa);                                     // np.round(...).astype(int)
                kb = __float2int_rn(qb);
                const uint32_t e = table_lookup(adv_t0, adv_t1, adv_t2, fsp * 10 + fbp * 5 + inv + 2);
                ka = max(min(ka, K_CLAMP), -K_CLAMP) + (int)(e & 3u) - 1;    // market_env.py:26-28
                kb = max(min(kb, K_CLAMP), -K_CLAMP) + (int)(e >> 2) - 1;
                fb = (inv2 < 1.0f) && (kb < kb1);                            // :34,:37
                fs = (inv2 > -1.0f) && (ka < ka1);                           // :35,:38
                fbp = fb ? 1 : 0; fsp = fs ? 1 : 0;                          // drl_engine.py:57-58
            } else {
                // rounding folded into the per-bar float threshold: no conversion on the critical path
                fb = (inv2 < 1.0f) && (qb < thb);
                fs = (inv2 > -1.0f) && (qa < tha);
            }
            inv2 = __fadd_rn(inv2, fb ? (fs ? 0.0f : 0.5f) : (fs ? -0.5f : 0.0f));   // :45,:51 (exact)
            inv += (fb ? 1 : 0) - (fs ? 1 : 0);
            // ---- step code: the offset of each side that filled -------------------------------
            if (l == 0) {
                if (ADV) *reinterpret_cast<int2*>(recs + i * 32) = make_int2(fs ? ka : SGMM_CODE_NOFILL, fb ? kb : SGMM_CODE_NOFILL);
                else *reinterpret_cast<float2*>(recs + i * 32) = make_float2(fs ? qa : __int_as_float(SGMM_CODE_NOFILL_F), fb ? qb : __int_as_float(SGMM_CODE_NOFILL_F));
            }
#pragma unroll
            for (int u = 0; u < U; ++u) A1[u] = A1n[u];
        }
        __syncwarp();
        if (lane == 0) { mbar_arrive(&sm.empty[s]); mbar_arrive(&sm.rec_full[r]); }
#ifdef SGMM_ROLLOUT_TRACE
        if (trc) for (int i = 0; i < 64; ++i)
            printf("w%d step %2d top %6lld burst_end %6lld reduced %6lld\n", warp, i, sm.trace[warp >> 2][i][0] - sm.trace[0][0][0],
                   sm.trace[warp >> 2][i][1] - sm.trace[0][0][0], sm.trace[warp >> 2][i][2] - sm.trace[0][0][0]);
#endif
    }
}


template <int U, bool ADV, bool FEE>
static int launch_variant(const RolloutArgs& args, int warps, cudaStream_t st)
{
    auto kern = rollout_kernel_h32<U, ADV, FEE>;
    static std::atomic<uint64_t> configured{0};   // per instantiation, one bit per device
    const size_t smem = sizeof(RingSmem);
    if (int rc = opt_in_smem(kern, smem, configured, "cudaFuncSetAttribute(smem)")) return rc;
    const int64_t per_cta = (int64_t)warps * U;
    const int64_t blocks = (args.mm.count + per_cta - 1) / per_cta;
    kern<<<(unsigned)blocks, (warps + 1) * 32, smem, st>>>(args);   // + the producer warp
    return check_cuda(cudaGetLastError(), "rollout_kernel_h32 launch");
}

template <int U>
static int launch_u(const RolloutArgs& args, bool adv, bool fee, int warps, cudaStream_t st)
{
    if (adv) return fee ? launch_variant<U, true, true>(args, warps, st) : launch_variant<U, true, false>(args, warps, st);
    return fee ? launch_variant<U, false, true>(args, warps, st) : launch_variant<U, false, false>(args, warps, st);
}

static int g_sm_count[64] = {0};

int launch_rollout(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, int hidden,
                   double phi, double fee, int units_per_lane, int warps_per_cta,
                   double* fitness, int32_t* trades, cudaStream_t st)
{
    if (hidden != 32) { set_error("hidden=%d: the SGMM-F32 rollout kernel is built for H=32", hidden); return SGMM_ERR_UNSUPPORTED; }
    if (mm.count == 0) return SGMM_OK;
    // small populations without an adversary: the policy-table path (sgmm_one.cu) unless the caller pinned a geometry
    {
        static const int64_t small_max = [] { const char* e = getenv("SGMM_SMALL_POP_MAX"); return e ? (int64_t)atoll(e) : SMALL_POP_MAX; }();
        static const int64_t small_max_adv = [] { const char* e = getenv("SGMM_SMALL_POP_MAX_ADV"); return e ? (int64_t)atoll(e) : SMALL_POP_MAX_ADV; }();
        // (with the adversary the walk kernel runs one CTA per SM: beyond the SM count it only wins on episodes of ~4+ days)
        const int64_t adv_max = b->T >= 900 ? 2 * small_max_adv : small_max_adv;
        if (units_per_lane == 0 && warps_per_cta == 0 && mm.count <= (adv ? adv_max : small_max))
            return launch_rollout_small(b, mm, adv, phi, fee, fitness, trades, st);
    }
    int dev = b->device;
    if (dev >= 0 && dev < 64 && g_sm_count[dev] == 0) {
        int n = 0;
        if (int rc = check_cuda(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev), "query SM count")) return rc;
        g_sm_count[dev] = n;
    }
    const int sms = (dev >= 0 && dev < 64 && g_sm_count[dev] > 0) ? g_sm_count[dev] : 148;
    int U = units_per_lane;
    // auto: a whole warp per individual while that still leaves at most one compute warp per scheduler (the step of a
    // lone warp is latency-bound and shortest with 32 lanes per individual: P = 50 x 14 400 bars 2.49 instead of 2.87 ms,
    // P = 512 2.69 / 2.87), four individuals per warp beyond (P = 1024: 2.90 / 3.10 ms, P = 4096: 4.5 / 8.2)
    if (U == 0) U = (mm.count <= 4 * (int64_t)sms) ? 1 : 4;
    if (U != 1 && U != 2 && U != 4) { set_error("units_per_lane must be 0, 1, 2 or 4"); return SGMM_ERR_INVALID; }
    int W = warps_per_cta;
    if (W == 0) {
        // one CTA per SM per wave; spread the population evenly over the SMs of each wave
        const int max_w = max_compute_warps(U);
        const int64_t per_sm_full = (int64_t)max_w * U;
        const int64_t waves = (mm.count + per_sm_full * sms - 1) / (per_sm_full * sms);
        const int64_t per_sm = (mm.count + waves * sms - 1) / (waves * sms);
        W = (int)((per_sm + U - 1) / U);
        if (W < 1) W = 1;
        if (W > max_w) W = max_w;
    }
    if (W < 1 || W > max_compute_warps(U)) { set_error("warps_per_cta must be in 1..%d for units_per_lane=%d", max_compute_warps(U), U); return SGMM_ERR_INVALID; }
    RolloutArgs args;
    args.sig = b->sig; args.px = b->px; args.T = b->T; args.tick = b->tick; args.phi = phi; args.fee = fee;
    args.mm = mm;
    if (adv) args.adv = *adv; else { PopArgs z = {}; args.adv = z; }
    args.fitness = fitness; args.trades = trades;
    args.codes = nullptr;
    const bool has_fee = (fee != 0.0);
    switch (U) {
        case 1: return launch_u<1>(args, adv != nullptr, has_fee, W, st);
        case 2: return launch_u<2>(args, adv != nullptr, has_fee, W, st);
        default: return launch_u<4>(args, adv != nullptr, has_fee, W, st);
    }
}

// ---------------------------------------------------------------------------------------------
// trace kernel: ONE individual, one warp (lane = hidden unit), the literal step core of
// sgmm_step_core.h on the raw bounds, and one recorder row per step (Env/recorder.py:8-36).
// Also the teacher-forced replay (forced actions) used for bit-exact env parity.
// ---------------------------------------------------------------------------------------------
struct TraceArgs {
    const BarSig* sig; const BarPx* px; const double* bmax; const double* smin;
    int64_t T; double tick, phi, fee;
    const float* mm; const float* adv; const int32_t* forced; const int32_t* table;
    const float2* raw;       // [T][5] raw policy outputs of every (bar, inventory) (H = 256: sgmm_exact256.cu)
    sgmm_trace tr; double* fitness; int32_t* trades;
};

__global__ void __launch_bounds__(32, 1) trace_kernel_h32(const TraceArgs a)
{
    constexpr int H = 32;
    const int lane = threadIdx.x;
    GenomeSource src; src.seeded = false; src.row = a.mm; src.sigma = 0.f; src.seed = src.generation = src.individual = 0;
    float w1x = 0, w1y = 0, w1i = 0, b1 = 0, b2 = 0, w3a = 0, w3b = 0, b3a = 0, b3b = 0;
    float w2[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) w2[k] = 0.0f;
    if (a.mm) {
        const int j = lane;
        w1x = src.at(3 * j); w1y = src.at(3 * j + 1); w1i = src.at(3 * j + 2);
        b1 = src.at(3 * H + j); b2 = src.at(4 * H + H * H + j);
        w3a = src.at(5 * H + H * H + j); w3b = src.at(6 * H + H * H + j);
        b3a = src.at(7 * H + H * H); b3b = src.at(7 * H + H * H + 1);
#pragma unroll
        for (int k = 0; k < 32; ++k) w2[k] = src.at(4 * H + j * H + k);
    }
    uint32_t adv_entry = 5u;
    if (a.adv && lane < 20) {
        GenomeSource asrc = src; asrc.row = a.adv;
        adv_entry = adversary_entry(asrc, lane);
    }
    sgmm_env_state env;
    env.phi = a.phi; env.tick_size = a.tick; env.fee_rate = a.fee;
    env.inventory = 0; env.cash = 0.0; env.i_max = 2; env.i_min = -2;         // market_env.py:9-15
    double total = 0.0; int trades = 0; int fbp = 0, fsp = 0;
    double cum_fees = 0.0;                                                     // Env/recorder.py:49
    for (int64_t t = 0; t < a.T; ++t) {
        const BarSig sg = a.sig[t];
        const BarPx px = a.px[t];
        const float inv2 = (float)((int)env.inventory) * 0.5f;
        float ra = 0.0f, rb = 0.0f; int ka, kb;
        if (a.forced) { ka = a.forced[2 * t]; kb = a.forced[2 * t + 1]; }
        else if (a.table) { const int64_t r = (t * 5 + (int)env.inventory + 2) * 2; ka = a.table[r]; kb = a.table[r + 1]; }
        else if (a.raw) {
            const float2 r = a.raw[t * 5 + (int)env.inventory + 2];
            ra = r.x; rb = r.y;
            ka = __float2int_rn(__fmul_rn(ra, 5.0f));
            kb = __float2int_rn(__fmul_rn(rb, 5.0f));
        } else {
            float v = __fmaf_rn(w1x, sg.z1, b1);
            v = __fmaf_rn(w1y, sg.z2, v);
            v = __fmaf_rn(w1i, inv2, v);
            const float h1 = fmaxf(v, 0.0f);
            float c0 = b2, c1 = 0.0f, c2 = 0.0f, c3 = 0.0f;
#pragma unroll
            for (int k = 0; k < 32; k += 4) {
                c0 = __fmaf_rn(w2[k + 0], __shfl_sync(0xffffffffu, h1, k + 0), c0);
                c1 = __fmaf_rn(w2[k + 1], __shfl_sync(0xffffffffu, h1, k + 1), c1);
                c2 = __fmaf_rn(w2[k + 2], __shfl_sync(0xffffffffu, h1, k + 2), c2);
                c3 = __fmaf_rn(w2[k + 3], __shfl_sync(0xffffffffu, h1, k + 3), c3);
            }
            const float h2 = fmaxf(__fadd_rn(__fadd_rn(c0, c2), __fadd_rn(c1, c3)), 0.0f);
            ra = __fmul_rn(w3a, h2); rb = __fmul_rn(w3b, h2);
#pragma unroll
            for (int m = 16; m >= 1; m >>= 1) {
                ra = __fadd_rn(ra, __shfl_xor_sync(0xffffffffu, ra, m));
                rb = __fadd_rn(rb, __shfl_xor_sync(0xffffffffu, rb, m));
            }
            ra = __fadd_rn(ra, b3a); rb = __fadd_rn(rb, b3b);
            ka = __float2int_rn(__fmul_rn(ra, 5.0f));
            kb = __float2int_rn(__fmul_rn(rb, 5.0f));
        }
        int da = 0, db = 0;
        if (a.adv) {
            const int st = fsp * 10 + fbp * 5 + (int)env.inventory + 2;
            const uint32_t e = __shfl_sync(0xffffffffu, adv_entry, st);
            da = (int)(e & 3u) - 1; db = (int)(e >> 2) - 1;
        }
        sgmm_step_info info;
        env_step(env, (int64_t)ka + da, (int64_t)kb + db, px.mid_next, px.ask, px.bid, a.bmax[t], a.smin[t], info);
        total = add_rn(total, info.reward);
        fbp = info.fill_buy; fsp = info.fill_sell;
        trades += (info.fill_buy | info.fill_sell);
        if (lane == 0) {
            const sgmm_trace& tr = a.tr;
            if (tr.off_a) tr.off_a[t] = ka;
            if (tr.off_b) tr.off_b[t] = kb;
            if (tr.adv_a) tr.adv_a[t] = da;
            if (tr.adv_b) tr.adv_b[t] = db;
            if (tr.fill_buy) tr.fill_buy[t] = info.fill_buy;
            if (tr.fill_sell) tr.fill_sell[t] = info.fill_sell;
            if (tr.inventory) tr.inventory[t] = (int32_t)env.inventory;
            if (tr.cash) tr.cash[t] = env.cash;
            if (tr.reward) tr.reward[t] = info.reward;
            if (tr.pnl_reward) tr.pnl_reward[t] = info.pnl_reward;
            if (tr.inventory_reward) tr.inventory_reward[t] = info.inventory_reward;
            if (tr.fee_paid) tr.fee_paid[t] = info.fee_paid;
            if (tr.raw_a) tr.raw_a[t] = ra;
            if (tr.raw_b) tr.raw_b[t] = rb;
            // derived columns (Env/recorder.py:45-51); `mid` of a recorded row is the bar's mid_next (agent_trainer.py:153)
            cum_fees = add_rn(cum_fees, info.fee_paid);
            const double unreal = mul_rn((double)env.inventory, px.mid_next);
            if (tr.spread) tr.spread[t] = sub_rn(px.ask, px.bid);
            if (tr.wealth) tr.wealth[t] = add_rn(env.cash, unreal);
            if (tr.cum_reward) tr.cum_reward[t] = total;
            if (tr.skew) tr.skew[t] = kb - ka;
            if (tr.cum_fees) tr.cum_fees[t] = cum_fees;
            if (tr.unrealized_pnl) tr.unrealized_pnl[t] = unreal;
        }
    }
    total = episode_fitness(total, trades);
    if (lane == 0) {
        if (a.fitness) *a.fitness = total;
        if (a.trades) *a.trades = trades;
    }
}

int launch_trace(const sgmm_bundle* b, const float* mm_genome, int hidden, const float* adv_genome,
                 const int32_t* forced, const int32_t* table, double phi, double fee, const sgmm_trace* tr,
                 double* fitness, int32_t* trades, cudaStream_t st)
{
    if (hidden != 32 && hidden != 256) { set_error("hidden=%d: the trace is built for H=32 and H=256", hidden); return SGMM_ERR_UNSUPPORTED; }
    if (!mm_genome && !forced && !table) { set_error("trace needs a genome, forced actions or an inventory table"); return SGMM_ERR_INVALID; }
    TraceArgs a;
    a.sig = b->sig; a.px = b->px; a.bmax = b->bmax; a.smin = b->smin; a.T = b->T;
    a.tick = b->tick; a.phi = phi; a.fee = fee; a.mm = mm_genome; a.adv = adv_genome; a.forced = forced; a.table = table;
    a.raw = nullptr;
    if (tr) a.tr = *tr; else { sgmm_trace z = {}; a.tr = z; }
    a.fitness = fitness; a.trades = trades;
    if (hidden == 256) {
        // the policy of every (bar, inventory) first (exact H = 256 table, raw outputs), then the same trace kernel on it
        a.mm = nullptr;
        if (mm_genome && !forced && !table) {
            uint64_t* buf = nullptr;
            const int64_t words = 5 * b->T + genome_len(256) / 2;               // float2[T][5] + room for one staged genome, reserved
                                                                                 // whether or not the genome needs staging (269 KB)
            if (int rc = reserve_codes(b, b->T > 0 ? (words + b->T - 1) / b->T : 1, st, &buf)) return rc;
            CodesRelease release(b, st);
            float2* raw = reinterpret_cast<float2*>(buf);
            if (b->T > 0)
                if (int rc = launch_exact256_raw(b, mm_genome, raw, reinterpret_cast<float*>(buf + 5 * b->T), st)) return rc;
            a.raw = raw;
            trace_kernel_h32<<<1, 32, 0, st>>>(a);
            if (int rc = check_cuda(cudaGetLastError(), "trace_kernel_h32 launch")) return rc;
            return release.done();
        }
    }
    trace_kernel_h32<<<1, 32, 0, st>>>(a);
    return check_cuda(cudaGetLastError(), "trace_kernel_h32 launch");
}

}  // namespace sgmm
