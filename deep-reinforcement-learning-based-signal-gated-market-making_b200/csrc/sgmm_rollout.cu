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
// the pieces of the rollout kernels (H = 32)
// ---------------------------------------------------------------------------------------------
// compute warps per CTA (one more warp is the producer): bounded by the register file
__host__ __device__ constexpr int max_compute_warps(int U) { return U == 4 ? 7 : (U == 2 ? 15 : MAX_WARPS); }

// where a thread sits: a CTA has nwarps compute warps of U individuals each (L = 32 / U lanes per individual) and, last,
// the producer / accounting warp
template <int U>
struct H32Cta {
    int warp, lane, nwarps;
    int g, l;                 // the lane's individual within the warp, and its lane within the individual
    int live_warps;           // compute warps with at least one individual < count
    int64_t first, ind;       // the CTA's first individual, the lane's individual
    bool live;                // ind < count

    __device__ __forceinline__ explicit H32Cta(const int64_t& count)
    {
        warp = threadIdx.x >> 5; lane = threadIdx.x & 31;
        nwarps = (blockDim.x >> 5) - 1;
        g = lane / (32 / U); l = lane % (32 / U);
        first = (int64_t)blockIdx.x * nwarps * U;
        const int64_t remaining = count - first;
        live_warps = (int)(remaining >= (int64_t)nwarps * U ? nwarps : (remaining + U - 1) / U);
        ind = first + (int64_t)warp * U + g;
        live = ind < count;
    }
};

// one bar of the accounting warp: the fp64 half of the env step of this lane's individual from its step record `code`
// (the offset of each side that filled, or a no-fill marker; without the adversary the offsets travel as the fp32 q = raw*5)
template <bool ADV, bool FEE>
__device__ __forceinline__ void account_bar(uint64_t code, const BarPx* pxs, int i, double tick, double fee,
                                            const PenaltyTable& pen, int& inv, int& ntr, double& total)
{
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

// the lane's weights in registers (models/model.py:31-36 layout): hidden units l, l + L, ... of W1 / b1 / b2 / W2 rows / W3,
// and b3; zeros for a lane without an individual
template <int U>
struct H32Regs {
    float w1x[U], w1y[U], w1i[U], b1[U], b2[U], w3a[U], w3b[U];
    float2 w2[U][16];
    float b3a, b3b;
};

template <int U>
__device__ __forceinline__ void h32_load_weights(const PopArgs& mm, const H32Cta<U>& cta, H32Regs<U>& w)
{
    constexpr int H = 32, L = 32 / U;
    const GenomeSource src = make_source(resolve(mm), cta.live ? cta.ind : 0, (int64_t)H * H + 7 * H + 2);
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int j = cta.l + L * u;
        if (cta.live) {
            w.w1x[u] = src.at(3 * j + 0); w.w1y[u] = src.at(3 * j + 1); w.w1i[u] = src.at(3 * j + 2);
            w.b1[u] = src.at(3 * H + j);
            w.b2[u] = src.at(4 * H + H * H + j);
            w.w3a[u] = src.at(5 * H + H * H + j);
            w.w3b[u] = src.at(6 * H + H * H + j);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float v[4]; src.at4(4 * H + (int64_t)j * H + 4 * c, v);
                w.w2[u][2 * c] = make_float2(v[0], v[1]);
                w.w2[u][2 * c + 1] = make_float2(v[2], v[3]);
            }
        } else {
            w.w1x[u] = w.w1y[u] = w.w1i[u] = w.b1[u] = w.b2[u] = w.w3a[u] = w.w3b[u] = 0.0f;
#pragma unroll
            for (int c = 0; c < 16; ++c) w.w2[u][c] = make_float2(0.0f, 0.0f);
        }
    }
    w.b3a = cta.live ? src.at(7 * H + H * H) : 0.0f;
    w.b3b = cta.live ? src.at(7 * H + H * H + 1) : 0.0f;
}

// the adversary's displacement table of the lane's individual (drl_engine.py:42-48, models/model.py:40-50): 4 bits for
// each of the 20 states in t[0..2]; the L lanes of an individual split the states, then gather the whole table
template <int U>
__device__ __forceinline__ void h32_adv_table(const PopArgs& adv, const H32Cta<U>& cta, uint32_t t[3])
{
    constexpr int L = 32 / U;
    const GenomeSource asrc = make_source(resolve(adv), cta.live ? cta.ind : 0, (int64_t)1250);
    t[0] = t[1] = t[2] = 0u;
    for (int s = cta.l; s < 20; s += L) {
        const uint32_t e = cta.live ? adversary_entry(asrc, s) : 5u;
        t[s >> 3] |= e << ((s & 7) * 4);
    }
#pragma unroll
    for (int m = L / 2; m >= 1; m >>= 1) {
#pragma unroll
        for (int k = 0; k < 3; ++k) t[k] |= __shfl_xor_sync(0xffffffffu, t[k], m);
    }
}

// layer 1 of one bar: the bar part w1x*z1 + w1y*z2 + b1 (inventory-independent), then the inventory term and the ReLU
template <int U>
__device__ __forceinline__ void h32_layer1_bar(const H32Regs<U>& w, float2 z, float a1[U])
{
#pragma unroll
    for (int u = 0; u < U; ++u) a1[u] = __fmaf_rn(w.w1y[u], z.y, __fmaf_rn(w.w1x[u], z.x, w.b1[u]));
}
template <int U>
__device__ __forceinline__ void h32_layer1_inv(const H32Regs<U>& w, const float a1[U], float inv2, float h[U])
{
#pragma unroll
    for (int u = 0; u < U; ++u) h[u] = fmaxf(__fmaf_rn(w.w1i[u], inv2, a1[u]), 0.0f);
}
template <int U>
__device__ __forceinline__ void h32_layer1(const H32Regs<U>& w, float2 z, float inv2, float h[U])
{
    float a1[U];
    h32_layer1_bar<U>(w, z, a1);
    h32_layer1_inv<U>(w, a1, inv2, h);
}
// h1 through the warp's shared buffer: U individuals x 32 activations, 16-B interleaved
template <int U>
__device__ __forceinline__ void h32_put_h1(float* hb, int g, int l, const float h[U])
{
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int j = l + (32 / U) * u;
        hb[((j >> 2) * U + g) * 4 + (j & 3)] = h[u];
    }
}
template <int U>
__device__ __forceinline__ void h32_get_h1(const float* hb, int g, float4 h4[8])
{
#pragma unroll
    for (int k = 0; k < 8; ++k) h4[k] = *reinterpret_cast<const float4*>(&hb[(k * U + g) * 4]);
}
// layers 2 and 3 up to the lane's partial outputs: U rows x 32 as packed FFMA2, four chains per row (the two halves of
// P and Q are the four interleaved chains of the SGMM-F32 order), then the products and the local tree; for U < 4 the
// cross-lane butterfly too (shuffles)
template <int U>
__device__ __forceinline__ float2 h32_layer23(const H32Regs<U>& w, const float4 h4[8])
{
    constexpr int L = 32 / U;
    float2 P[U], Q[U];
#pragma unroll
    for (int u = 0; u < U; ++u) { P[u] = make_float2(w.b2[u], 0.0f); Q[u] = make_float2(0.0f, 0.0f); }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float2 hlo = make_float2(h4[k].x, h4[k].y), hhi = make_float2(h4[k].z, h4[k].w);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            P[u] = __ffma2_rn(w.w2[u][2 * k], hlo, P[u]);
            Q[u] = __ffma2_rn(w.w2[u][2 * k + 1], hhi, Q[u]);
        }
    }
    float pa[U], pb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const float2 S = __fadd2_rn(P[u], Q[u]);                 // (a0+a2, a1+a3)
        const float h2 = fmaxf(__fadd_rn(S.x, S.y), 0.0f);
        pa[u] = __fmul_rn(w.w3a[u], h2);
        pb[u] = __fmul_rn(w.w3b[u], h2);
    }
    float ra, rb;
    if (U == 4) {
        ra = __fadd_rn(__fadd_rn(pa[0], pa[2 % U]), __fadd_rn(pa[1 % U], pa[3 % U]));
        rb = __fadd_rn(__fadd_rn(pb[0], pb[2 % U]), __fadd_rn(pb[1 % U], pb[3 % U]));
    } else {
        if (U == 2) { ra = __fadd_rn(pa[0], pa[1 % U]); rb = __fadd_rn(pb[0], pb[1 % U]); }
        else { ra = pa[0]; rb = pb[0]; }
#pragma unroll
        for (int m = L / 2; m >= 1; m >>= 1) {
            ra = __fadd_rn(ra, __shfl_xor_sync(0xffffffffu, ra, m));
            rb = __fadd_rn(rb, __shfl_xor_sync(0xffffffffu, rb, m));
        }
    }
    return make_float2(ra, rb);
}
// U = 4: the butterfly over the 8 lanes of the individual, evaluated by every lane from the 8 partials exchanged through
// shared memory (the same tree, one round trip instead of 3 shuffles)
__device__ __forceinline__ void h32_put_partial(float* rbw, int g, int l, float2 r)
{
    *reinterpret_cast<float2*>(&rbw[g * 20 + l * 2]) = r;
}
__device__ __forceinline__ void h32_get_partials(const float* rbw, int g, float4 r[4])
{
#pragma unroll
    for (int k = 0; k < 4; ++k) r[k] = *reinterpret_cast<const float4*>(&rbw[g * 20 + 4 * k]);
}
__device__ __forceinline__ float2 h32_tree(const float4 r[4])
{
    const float2 t04 = __fadd2_rn(make_float2(r[0].x, r[0].y), make_float2(r[2].x, r[2].y));
    const float2 t15 = __fadd2_rn(make_float2(r[0].z, r[0].w), make_float2(r[2].z, r[2].w));
    const float2 t26 = __fadd2_rn(make_float2(r[1].x, r[1].y), make_float2(r[3].x, r[3].y));
    const float2 t37 = __fadd2_rn(make_float2(r[1].z, r[1].w), make_float2(r[3].z, r[3].w));
    return __fadd2_rn(__fadd2_rn(t04, t26), __fadd2_rn(t15, t37));
}
// layers 2 and 3 of one chain from the h1 it published: the individual's raw outputs before b3
template <int U>
__device__ __forceinline__ float2 h32_output(const H32Regs<U>& w, const float* hb, float* rbw, int g, int l)
{
    float4 h4[8];
    h32_get_h1<U>(hb, g, h4);
    float2 p = h32_layer23<U>(w, h4);
    if (U == 4) {
        h32_put_partial(rbw, g, l, p);
        __syncwarp();
        float4 pr[4];
        h32_get_partials(rbw, g, pr);
        p = h32_tree(pr);
    }
    return p;
}

// the fill decision: q = raw*5 (drl_engine.py:39), and the inventory move (in halves, exact) of the fills
__device__ __forceinline__ float2 h32_q(float2 r, float b3a, float b3b)
{
    return make_float2(__fmul_rn(__fadd_rn(r.x, b3a), 5.0f), __fmul_rn(__fadd_rn(r.y, b3b), 5.0f));
}
__device__ __forceinline__ float h32_move(bool fb, bool fs) { return fb ? (fs ? 0.0f : 0.5f) : (fs ? -0.5f : 0.0f); }   // market_env.py:45,51
// without the adversary: the rounding is folded into the bar's float thresholds th = (tha, thb), so there is no
// conversion on the critical path; moves inv2 and returns the step record (the q of each side that filled)
__device__ __forceinline__ float2 h32_decide(float2 r, float b3a, float b3b, float2 th, float& inv2)
{
    const float2 q = h32_q(r, b3a, b3b);
    const bool fb = (inv2 < 1.0f) && (q.y < th.y);                 // market_env.py:34,37
    const bool fs = (inv2 > -1.0f) && (q.x < th.x);                // :35,:38
    inv2 = __fadd_rn(inv2, h32_move(fb, fs));
    return make_float2(fs ? q.x : __int_as_float(SGMM_CODE_NOFILL_F), fb ? q.y : __int_as_float(SGMM_CODE_NOFILL_F));
}
// with the adversary (drl_engine.py:42-48): integer offsets, clamped and displaced by the table entry of the state
// (previous fills, inventory), against the bar's integer thresholds k1 = (ka1, kb1); moves the state and returns the step
// record (the offset of each side that filled)
__device__ __forceinline__ int2 h32_decide_adv(float2 r, float b3a, float b3b, int2 k1, const uint32_t t[3], int& inv,
                                               int& fbp, int& fsp, float& inv2)
{
    const float2 q = h32_q(r, b3a, b3b);
    int ka = __float2int_rn(q.x), kb = __float2int_rn(q.y);        // np.round(...).astype(int)
    const uint32_t e = table_lookup(t[0], t[1], t[2], fsp * 10 + fbp * 5 + inv + 2);
    ka = max(min(ka, K_CLAMP), -K_CLAMP) + (int)(e & 3u) - 1;      // market_env.py:26-28
    kb = max(min(kb, K_CLAMP), -K_CLAMP) + (int)(e >> 2) - 1;
    const bool fb = (inv2 < 1.0f) && (kb < k1.y);                  // :34,:37
    const bool fs = (inv2 > -1.0f) && (ka < k1.x);                 // :35,:38
    fbp = fb ? 1 : 0; fsp = fs ? 1 : 0;                            // drl_engine.py:57-58
    inv2 = __fadd_rn(inv2, h32_move(fb, fs));
    inv += (fb ? 1 : 0) - (fs ? 1 : 0);
    return make_int2(fs ? ka : SGMM_CODE_NOFILL, fb ? kb : SGMM_CODE_NOFILL);
}
// the inventory move (in halves) a step record of h32_decide encodes
__device__ __forceinline__ float h32_record_move(float2 c)
{
    return h32_move(__float_as_int(c.y) != SGMM_CODE_NOFILL_F, __float_as_int(c.x) != SGMM_CODE_NOFILL_F);
}

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
};

template <int U, bool ADV, bool FEE>
__global__ void __launch_bounds__((max_compute_warps(U) + 1) * 32, 1)
rollout_kernel_h32(const RolloutArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    RingSmem& sm = *reinterpret_cast<RingSmem*>(smem_raw);

    const H32Cta<U> cta(a.mm.count);
    const int64_t T = a.T;
    const int64_t nchunks = (T + CHUNK_BARS - 1) / CHUNK_BARS;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < RING_STAGES; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], cta.live_warps); }
#pragma unroll
        for (int r = 0; r < REC_STAGES; ++r) { mbar_init(&sm.rec_full[r], cta.live_warps); mbar_init(&sm.rec_empty[r], 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (cta.warp == cta.nwarps) {
        // ===== the CTA's last warp: TMA producer of the bar ring AND the fp64 half of the env step =====
        // The compute warps do the policy and the INTEGER half of the step and hand one 8-byte record per bar and
        // individual through shared memory; here lane j accounts individual first + j: quotes, P&L legs, penalty and
        // the bar-order reward sum in the reference's un-fused fp64 (market_env.py:30-58, drl_engine.py:54).  One
        // warp instruction per fp64 operation for ALL individuals of the CTA -- in the step loop the same arithmetic
        // was issued once per compute warp (22 of 217 instructions, two of them conversions on the XU pipe, plus the
        // fp64 live ranges in a 254-register kernel) and cost 16 % of the loop.
        const int lane = cta.lane;
        const int64_t indj = cta.first + lane;
        const bool livej = lane < cta.live_warps * U && indj < a.mm.count;
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
                account_bar<ADV, FEE>(sm.rec[r][i][lane], pxs, i, tick, fee, pen, inv, ntr, total);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.rec_empty[r]);
        }
        if (livej) { a.fitness[indj] = episode_fitness(total, ntr); a.trades[indj] = ntr; }
        return;
    }
    if (cta.warp >= cta.live_warps) return;

    H32Regs<U> w;
    h32_load_weights<U>(a.mm, cta, w);
    uint32_t adv_t[3] = {0u, 0u, 0u};
    if (ADV) h32_adv_table<U>(a.adv, cta, adv_t);

    float* const hb = &sm.hbuf[cta.warp][0];
    float* const rbw = &sm.rbuf[cta.warp][0];
    int inv = 0, fbp = 0, fsp = 0;                                   // the adversary's state
    float inv2 = 0.0f;                                               // inventory / 2.0 (drl_engine.py:35), exact

    // The step loop does the INTEGER half of the env step (offsets, fills, inventory) and hands one 8-byte record per
    // bar to the accounting warp (above).
    const int slotj = cta.warp * U + cta.g;                          // this individual's lane in the accounting warp

    // Two compute warps share a scheduler (warps w and w + 4).  Measured (profiles/r2_exact_phase_trace_*.log, a clock64 trace of
    // both from a trace build, removed after 2e97c64): their steps lock at a relative phase of 0.19 whatever the start offset, and
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

        // bar 0 of the chunk: signals, thresholds and the bar part of layer 1
        float4 sg = *reinterpret_cast<const float4*>(&sigs[0]);                     // z1, z2, tha, thb
        int2 kth = *reinterpret_cast<const int2*>(&sigs[0].ka1);
        float a1[U];
        h32_layer1_bar<U>(w, make_float2(sg.x, sg.y), a1);
#pragma unroll 1
        for (int i = 0; i < n; ++i) {
            float h[U];
            h32_layer1_inv<U>(w, a1, inv2, h);
            h32_put_h1<U>(hb, cta.g, cta.l, h);
            __syncwarp();
            const float2 th = make_float2(sg.z, sg.w);
            const int2 k1 = kth;
            const float2 p = h32_output<U>(w, hb, rbw, cta.g, cta.l);
            // prefetch bar i+1 and the bar part of its layer 1 (off the critical path)
            const int inext = i + 1 < CHUNK_BARS ? i + 1 : CHUNK_BARS - 1;
            sg = *reinterpret_cast<const float4*>(&sigs[inext]);
            if (ADV) kth = *reinterpret_cast<const int2*>(&sigs[inext].ka1);
            h32_layer1_bar<U>(w, make_float2(sg.x, sg.y), a1);
            if (ADV) {
                const int2 code = h32_decide_adv(p, w.b3a, w.b3b, k1, adv_t, inv, fbp, fsp, inv2);
                if (cta.l == 0) *reinterpret_cast<int2*>(recs + i * 32) = code;
            } else {
                const float2 code = h32_decide(p, w.b3a, w.b3b, th, inv2);
                if (cta.l == 0) *reinterpret_cast<float2*>(recs + i * 32) = code;
            }
        }
        __syncwarp();
        if (cta.lane == 0) { mbar_arrive(&sm.empty[s]); mbar_arrive(&sm.rec_full[r]); }
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

// ---------------------------------------------------------------------------------------------
// the two-chain rollout kernel (H = 32, no adversary)
// ---------------------------------------------------------------------------------------------
// rollout_kernel_h32 advances one dependent chain per individual, and two warps per scheduler cannot hide it (§5 of
// DESIGN.md: ~620 cycles per pair of warp-steps, ~400 of them FMA-pipe time).  Here every warp advances TWO time blocks
// of its individuals' episodes on the same weight registers.  The episode runs in rounds of ROUND_BARS bars; with a
// burn-in of B bars and N = (ROUND_BARS + B) / 2:
//   * chain A steps bars [0, N) of the round from the exact state the previous round left;
//   * chain B steps bars [N - B, ROUND_BARS) from inventory 0; its first B bars are burn-in.
// Without the adversary the state entering a bar is the inventory alone, and a step's record is a function of (bar,
// inventory): once B's inventory equals the true one, B's records are the true records.  At the round's end each
// individual compares A's inventory entering bar N with B's; where they differ, B's block is stepped again from the
// true state (warp-uniform loop, lone chain) until the repaired inventory meets B's, or to the round's end.  Cold
// starts join fast (tools/exact_join_stats.py: median 3 bars; after 8 bars 10 % have not, after 16 bars 2.1 %);
// the path is exact for a policy that never joins.  A partial last round runs chain A alone.
// Measured on one B200 (1 000 W, profiles/r8_exact_chains_bench.json): P = 592 (U = 1, one warp per scheduler) 2.16 instead
// of 2.68 ms; P = 4096 (U = 4, two warps per scheduler) only 4.35 instead of 4.51 ms -- there the two warps already
// overlap most of each other's chain.  Loading half of the burst's activations after the other chain's stores (which
// moves its decision in front of the burst in the SASS) was slower: 4.60 ms at P = 4096, 2.68 ms at P = 592.
// The accounting warp consumes whole validated rounds in bar order: two round buffers of records and bars (the round
// r + 2 is loaded once round r is accounted), so the fp64 reward sum keeps the reference's order.
constexpr int ROUND_BARS = 256;
constexpr int ROLLOUT_BURN_IN = 4;        // default burn-in of chain B (even, < ROUND_BARS): 4.350 ms at the bench shape, 8: 4.379, 16: 4.44, 32: 4.66

struct Ring2Smem {
    uint64_t full[2];                     // the round's bars landed (TMA)
    uint64_t rec_full[2];                 // the round's records are validated (one arrival per compute warp)
    BarSig sig[2][ROUND_BARS];
    BarPx px[2][ROUND_BARS];              // prices: read by the accounting warp only
    float hbuf[2][MAX_WARPS][128];        // [chain][warp]: as RingSmem::hbuf
    float rbuf[2][MAX_WARPS][80];         // [chain][warp]: as RingSmem::rbuf
    uint64_t rec[2][ROUND_BARS][32];      // one 8-byte step record per (bar of the round, individual of the CTA)
};

template <int U, bool FEE>
__global__ void __launch_bounds__((max_compute_warps(U) + 1) * 32, 1)
rollout2_kernel_h32(const RolloutArgs a, const int burn)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Ring2Smem& sm = *reinterpret_cast<Ring2Smem*>(smem_raw);

    const H32Cta<U> cta(a.mm.count);
    const int64_t T = a.T;
    const int64_t nrounds = (T + ROUND_BARS - 1) / ROUND_BARS;
    const int N = (ROUND_BARS + burn) / 2;                           // steps of each chain in a whole round

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < 2; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.rec_full[s], cta.live_warps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (cta.warp == cta.nwarps) {
        // ===== TMA producer of the round buffers and the fp64 half of the env step (as in rollout_kernel_h32) =====
        const int lane = cta.lane;
        const int64_t indj = cta.first + lane;
        const bool livej = lane < cta.live_warps * U && indj < a.mm.count;
        const double tick = a.tick, fee = a.fee;
        const PenaltyTable pen = penalty_table(a.phi);
        double total = 0.0;
        int ntr = 0, inv = 0;
        auto load = [&](int64_t r) {
            if (lane == 0) {
                const int s = (int)(r & 1);
                const int64_t tl = r * ROUND_BARS;
                const uint32_t nb = (uint32_t)(T - tl < ROUND_BARS ? T - tl : ROUND_BARS);
                mbar_arrive_expect_tx(&sm.full[s], nb * (uint32_t)(sizeof(BarSig) + sizeof(BarPx)));
                tma_bulk_g2s(&sm.sig[s][0], a.sig + tl, nb * (uint32_t)sizeof(BarSig), &sm.full[s]);
                tma_bulk_g2s(&sm.px[s][0], a.px + tl, nb * (uint32_t)sizeof(BarPx), &sm.full[s]);
            }
        };
        for (int64_t r = 0; r < nrounds && r < 2; ++r) load(r);
        for (int64_t r = 0; r < nrounds; ++r) {
            const int s = (int)(r & 1);
            mbar_wait(&sm.rec_full[s], (uint32_t)((r >> 1) & 1));
            const int64_t t0 = r * ROUND_BARS;
            const int n = (int)(T - t0 < ROUND_BARS ? T - t0 : ROUND_BARS);
            const BarPx* pxs = &sm.px[s][0];
#pragma unroll 4
            for (int i = 0; i < n; ++i) {
                account_bar<false, FEE>(sm.rec[s][i][lane], pxs, i, tick, fee, pen, inv, ntr, total);
            }
            __syncwarp();
            if (r + 2 < nrounds) load(r + 2);                            // both buffers of round r are free again
        }
        if (livej) { a.fitness[indj] = episode_fitness(total, ntr); a.trades[indj] = ntr; }
        return;
    }
    if (cta.warp >= cta.live_warps) return;

    H32Regs<U> w;
    h32_load_weights<U>(a.mm, cta, w);

    float* const hA = &sm.hbuf[0][cta.warp][0];
    float* const hB = &sm.hbuf[1][cta.warp][0];
    float* const rA = &sm.rbuf[0][cta.warp][0];
    float* const rB = &sm.rbuf[1][cta.warp][0];
    const int slotj = cta.warp * U + cta.g;                         // this individual's lane in the accounting warp
    float inv2 = 0.0f;                                               // inventory / 2.0 (drl_engine.py:35), exact

    // one step of a lone chain on chain A's buffers (partial rounds and repairs); returns the step record
    auto step1 = [&](const BarSig* sg, float& iv) -> float2 {
        float h[U];
        h32_layer1<U>(w, *reinterpret_cast<const float2*>(&sg->z1), iv, h);
        h32_put_h1<U>(hA, cta.g, cta.l, h);
        __syncwarp();
        return h32_decide(h32_output<U>(w, hA, rA, cta.g, cta.l), w.b3a, w.b3b, *reinterpret_cast<const float2*>(&sg->tha), iv);
    };

    for (int64_t r = 0; r < nrounds; ++r) {
        const int s = (int)(r & 1);
        mbar_wait(&sm.full[s], (uint32_t)((r >> 1) & 1));               // also: round r - 2 is accounted
        __syncwarp();
        const BarSig* const sigs = &sm.sig[s][0];
        float2* const recs = reinterpret_cast<float2*>(&sm.rec[s][0][slotj]);   // bar i at recs[32 * i]
        const int64_t t0 = r * ROUND_BARS;
        const int n = (int)(T - t0 < ROUND_BARS ? T - t0 : ROUND_BARS);

        if (n < ROUND_BARS) {
#pragma unroll 1
            for (int i = 0; i < n; ++i) recs[32 * i] = step1(&sigs[i], inv2);
        } else {
            // ---- two chains.  B runs half a step behind A: each half-step overlaps one chain's layer-2 burst with
            // the other's reduction, fill decision and next layer 1; all loads of a half come first in program order,
            // its stores last, so that ptxas can interleave the two chains' arithmetic.
            const BarSig* const sigB = sigs + (N - burn);
            float2* const recB = recs + 32 * (N - burn);     // burn-in records land on bars chain A rewrites later
            float inv2B = 0.0f, inv2Bent = 0.0f;           // B's inventory; B's inventory entering bar N
            float2 pA, pB;
            {
                float h[U];
                h32_layer1<U>(w, *reinterpret_cast<const float2*>(&sigs[0].z1), inv2, h);
                h32_put_h1<U>(hA, cta.g, cta.l, h);
                h32_layer1<U>(w, *reinterpret_cast<const float2*>(&sigB[0].z1), inv2B, h);
                h32_put_h1<U>(hB, cta.g, cta.l, h);
                __syncwarp();
                float4 h4[8];
                h32_get_h1<U>(hB, cta.g, h4);
                pB = h32_layer23<U>(w, h4);
                if (U == 4) h32_put_partial(rB, cta.g, cta.l, pB);
            }
#pragma unroll 1
            for (int i = 0; i < N; ++i) {
                const int ibn = N - burn + i + 1 < ROUND_BARS ? i + 1 : i;   // B's next bar (the last one is not used)
                // -- half 1: A's layer 2 of bar i | B's decision of its bar i and layer 1 of the next
                __syncwarp();
                {
                    float4 h4[8];
                    h32_get_h1<U>(hA, cta.g, h4);
                    float2 qB = pB;
                    if (U == 4) { float4 pr[4]; h32_get_partials(rB, cta.g, pr); qB = h32_tree(pr); }
                    const float2 thB = *reinterpret_cast<const float2*>(&sigB[i].tha);
                    const float2 zB = *reinterpret_cast<const float2*>(&sigB[ibn].z1);
                    const float2 cB = h32_decide(qB, w.b3a, w.b3b, thB, inv2B);
                    inv2Bent = i == burn - 1 ? inv2B : inv2Bent;
                    float h[U];
                    h32_layer1<U>(w, zB, inv2B, h);
                    pA = h32_layer23<U>(w, h4);
                    recB[32 * i] = cB;
                    h32_put_h1<U>(hB, cta.g, cta.l, h);
                    if (U == 4) h32_put_partial(rA, cta.g, cta.l, pA);
                }
                // -- half 2: B's layer 2 of its next bar | A's decision of bar i and layer 1 of bar i + 1
                __syncwarp();
                {
                    float4 h4[8];
                    h32_get_h1<U>(hB, cta.g, h4);
                    float2 qA = pA;
                    if (U == 4) { float4 pr[4]; h32_get_partials(rA, cta.g, pr); qA = h32_tree(pr); }
                    const float2 thA = *reinterpret_cast<const float2*>(&sigs[i].tha);
                    const float2 zA = *reinterpret_cast<const float2*>(&sigs[i + 1].z1);    // i + 1 <= N < ROUND_BARS
                    const float2 cA = h32_decide(qA, w.b3a, w.b3b, thA, inv2);
                    float h[U];
                    h32_layer1<U>(w, zA, inv2, h);
                    pB = h32_layer23<U>(w, h4);
                    recs[32 * i] = cA;
                    h32_put_h1<U>(hA, cta.g, cta.l, h);
                    if (U == 4) h32_put_partial(rB, cta.g, cta.l, pB);
                }
            }
            __syncwarp();
            // ---- stitch: where B entered bar N with another inventory than A left it, step B's block again from the
            // true state until the two inventories meet (from there on the records are the same) or the block ends.
            // B's own inventory entering each bar comes from the record about to be overwritten.
            bool fix = cta.live && inv2 != inv2Bent;
            float inv2R = inv2, inv2O = inv2Bent;
#pragma unroll 1
            for (int j = N; j < ROUND_BARS && __any_sync(0xffffffffu, fix); ++j) {
                const float2 old = recs[32 * j];                                // read before step1's __syncwarp
                const float2 c = step1(&sigs[j], inv2R);
                inv2O = __fadd_rn(inv2O, h32_record_move(old));
                recs[32 * j] = fix ? c : old;
                fix = fix && inv2R != inv2O;
            }
            inv2 = fix ? inv2R : inv2B;                                         // the state entering the next round
        }
        __syncwarp();
        if (cta.lane == 0) mbar_arrive(&sm.rec_full[s]);
    }
}

template <int U, bool FEE>
static int launch_variant2(const RolloutArgs& args, int warps, int burn, cudaStream_t st)
{
    auto kern = rollout2_kernel_h32<U, FEE>;
    static std::atomic<uint64_t> configured{0};   // per instantiation, one bit per device
    const size_t smem = sizeof(Ring2Smem);
    if (int rc = opt_in_smem(kern, smem, configured, "cudaFuncSetAttribute(smem)")) return rc;
    const int64_t per_cta = (int64_t)warps * U;
    const int64_t blocks = (args.mm.count + per_cta - 1) / per_cta;
    kern<<<(unsigned)blocks, (warps + 1) * 32, smem, st>>>(args, burn);   // + the producer warp
    return check_cuda(cudaGetLastError(), "rollout2_kernel_h32 launch");
}

template <int U>
static int launch_u2(const RolloutArgs& args, bool fee, int warps, int burn, cudaStream_t st)
{
    return fee ? launch_variant2<U, true>(args, warps, burn, st) : launch_variant2<U, false>(args, warps, burn, st);
}

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
    const int sms = sm_count(b->device);
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
    // without the adversary: two time blocks per warp (rollout2_kernel_h32) unless SGMM_ROLLOUT_CHAINS=1; the burn-in of
    // the second block from SGMM_ROLLOUT_BURN_IN (even, 0 .. ROUND_BARS - 2; 0 makes the stitch repair almost every round)
    static const int chains = [] { const char* e = getenv("SGMM_ROLLOUT_CHAINS"); return e && atoi(e) == 1 ? 1 : 2; }();
    static const int burn = [] {
        const char* e = getenv("SGMM_ROLLOUT_BURN_IN");
        const int v = e ? atoi(e) : ROLLOUT_BURN_IN;
        return (v < 0 ? 0 : (v > ROUND_BARS - 2 ? ROUND_BARS - 2 : v)) & ~1;
    }();
    // (U = 2, only when pinned by the caller, stays single-chain: 5.49 against 5.35 ms at P = 4096 x 14 400 bars)
    if (!adv && chains == 2 && U != 2) return U == 1 ? launch_u2<1>(args, has_fee, W, burn, st) : launch_u2<4>(args, has_fee, W, burn, st);
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
            ScratchLease lease(b, st);
            uint64_t* buf = nullptr;
            // float2[T][5] + room for one staged genome, reserved whether or not the genome needs staging (269 KB)
            if (int rc = lease.reserve(5 * b->T + genome_len(256) / 2, &buf)) return rc;
            float2* raw = reinterpret_cast<float2*>(buf);
            if (b->T > 0)
                if (int rc = launch_exact256_raw(b, mm_genome, raw, reinterpret_cast<float*>(buf + 5 * b->T), st)) return rc;
            a.raw = raw;
            trace_kernel_h32<<<1, 32, 0, st>>>(a);
            if (int rc = check_cuda(cudaGetLastError(), "trace_kernel_h32 launch")) return rc;
            return lease.done();
        }
    }
    trace_kernel_h32<<<1, 32, 0, st>>>(a);
    return check_cuda(cudaGetLastError(), "trace_kernel_h32 launch");
}

}  // namespace sgmm
