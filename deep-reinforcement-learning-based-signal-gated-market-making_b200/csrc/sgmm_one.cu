// sgmm_one.cu -- SMALL populations, fast: the validation rollout of a GA generation (Env/drl_engine.py:129-140: the
// generation's best child on the validation bundle, adversary off), a single evaluate_individual call, and populations
// of the reference's own size (pop_size = 50, Env/drl_engine.py:70).
//
// The population kernel gives an individual one warp (or eight lanes) and walks the bars one after the other: below a
// few hundred individuals that is a handful of latency-bound warps on an otherwise idle GPU (one individual x 2 880
// bars = 0.64 ms, 13 % of a 4096-individual generation; 50 individuals x 14 400 bars = 2.5 ms = 0.29 G env-steps/s).
// With no adversary the action at bar t depends on (t, inventory) only and the inventory has five values
// (SURVEY.md 7.3), so the episode splits into
//   1. policy_table_kernel  the exact policy (SGMM-F32 order: the operations of trace_kernel_h32 in the same order) for
//                           EVERY (bar, inventory) pair -- 5 T independent evaluations spread over the whole GPU, one pair
//                           per thread with the weights broadcast from shared memory -- and the integer half of the env
//                           step of the pair: fills, next inventory, 8-byte step code;
//   2. walk_account_kernel<Walk5>  one CTA: the walk through the 5-state automaton as a parallel prefix scan over function
//                           composition (every bar is a map {0..4} -> {0..4}; composition is associative), then the fp64
//                           half for the visited pairs in parallel, and the one thing that is inherently serial -- the
//                           reference-order fp64 reward sum (drl_engine.py:54) -- by one thread, chunk by chunk.
//                           With the adversary the same kernel walks a 20-state automaton (walk_account_kernel<Walk20>).
// 5x the policy FLOPs of the sequential walk, ~10x less time; results bit-identical to rollout_kernel_h32
// (tests/test_gpu_configs.py compares both with the oracle; the GA parity tests compare whole histories).  One CTA of
// walk_account_kernel per individual; the launcher takes this path below SMALL_POP_MAX individuals (measured break-even
// against the sequential kernel: profiles/r2_small_population_path.log).
#include <type_traits>
#include "sgmm_internal.h"
#include "sgmm_rng.cuh"
#include "sgmm_adversary.cuh"
#include "sgmm_step_core.h"
#include "sgmm_walk.cuh"
#include "sgmm_np_sum.cuh"

namespace sgmm {

namespace one {

constexpr int H = 32;
constexpr int SUM_CHUNK = 2048;            // bars whose rewards sit in shared memory while one thread sums them

struct Scratch {                           // per (bar, inventory index) pair, written by policy_table_kernel
    float2* code;                          // [T][5]  q = raw*5 of each side that filled, NaN marker otherwise
    uint8_t* next;                         // [T][8]  next inventory index (bytes 0..4)
};

constexpr int PT_THREADS = 128;           // policy_table_kernel: one (bar, inventory) pair per thread, one individual per block task

// The individual's weights as the block stages them in shared memory: per hidden unit j one float4 {W1[j,0], W1[j,1], W1[j,2],
// b1[j]}, W2 row-major, b2, W3 as float2 {W3[0,j], W3[1,j]}, b3.  Every lane reads the SAME address at a time (a broadcast:
// one wavefront per load), so the policy of 32 different pairs costs the shared-memory traffic of one.
struct PtSmem {
    float4 l1[H];
    float w2[H][H];
    float b2[H];
    float2 w3[H];
    float b3[2];
};

// (Bar, inventory) pairs per THREAD -- two at a time, so that every broadcast weight load feeds two fma chains -- with the
// individual's weights broadcast from shared memory: ~53 warp instructions per pair instead of the ~110 (42 of them
// shuffles) of a lane-per-hidden-unit mapping, FMA-pipe / shared-load bound instead of shuffle bound (measured: lane per
// hidden unit 2.5x slower, one pair per thread 1.15x slower than this).  Same operations in the same order as trace_kernel_h32 (SGMM-F32
// order): layer 1 fma chain from b1; layer 2 four chains over k mod 4 from (b2, 0, 0, 0), combined (c0+c2)+(c1+c3); layer 3
// products summed by the xor-butterfly tree 16, 8, 4, 2, 1 (written out serially: s[l] = s[l] + s[l + m]) plus b3.
// RAW_OUT: the table holds the raw outputs before x5 (the population trace, sgmm_trace_pop.cu), and `raw` is ignored; its
// launch bound lets ptxas take 180 registers instead of spilling two words at 168.
// Pop: PopArgs (a population), or SweepPop (the children of a GA sweep: individual i of the launch is child
// (mm.first + i) % lambda of run (mm.first + i) / lambda).
template <bool RAW_OUT, class Pop>
__global__ void __launch_bounds__(PT_THREADS, RAW_OUT ? 1 : 0) policy_table_kernel(const BarSig* __restrict__ sig, int64_t T, const Pop mm_in, int64_t pairs_per_task,
                                                                   int raw, float2* __restrict__ code, uint8_t* __restrict__ next)
{
    __shared__ PtSmem sm;
    const Pop mm = resolve(mm_in);
    constexpr int64_t G = (int64_t)H * H + 7 * H + 2;
    const int64_t pairs = T * 5, tasks_per_ind = (pairs + pairs_per_task - 1) / pairs_per_task, ntasks = mm.count * tasks_per_ind;
    int64_t loaded = -1;
    for (int64_t task = blockIdx.x; task < ntasks; task += gridDim.x) {
        const int64_t ind = task / tasks_per_ind;
        if (ind != loaded) {                                   // (consecutive tasks of a block usually belong to different individuals)
            __syncthreads();
            const GenomeSource src = make_source(mm, ind, G);
            for (int q = threadIdx.x; q < 313; q += PT_THREADS) {                 // genome in groups of four elements (models/model.py:31-36 layout)
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (q < 312) src.at4(4 * q, v); else { v[0] = src.at(1248); v[1] = src.at(1249); }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int e = 4 * q + i;
                    if (e < 96) reinterpret_cast<float*>(&sm.l1[e / 3])[e % 3] = v[i];                   // W1[j, i]
                    else if (e < 128) sm.l1[e - 96].w = v[i];                                              // b1[j]
                    else if (e < 1152) sm.w2[(e - 128) >> 5][(e - 128) & 31] = v[i];                       // W2[j, k]
                    else if (e < 1184) sm.b2[e - 1152] = v[i];
                    else if (e < 1248) reinterpret_cast<float*>(&sm.w3[(e - 1184) & 31])[(e - 1184) >> 5] = v[i];   // W3[o, j]
                    else if (e < 1250) sm.b3[e - 1248] = v[i];
                }
            }
            __syncthreads();
            loaded = ind;
        }
        const int64_t p_lo = (task - ind * tasks_per_ind) * pairs_per_task, p_hi = p_lo + pairs_per_task < pairs ? p_lo + pairs_per_task : pairs;
        float2* codei = code + ind * pairs;
        uint8_t* nexti = next + ind * T * 8;
        // TWO pairs per thread and round (p and p + PT_THREADS): every broadcast weight load feeds two fma chains
        for (int64_t p0 = p_lo + threadIdx.x; p0 < p_hi; p0 += 2 * PT_THREADS) {
            const int64_t pp[2] = {p0, p0 + PT_THREADS};
            const bool ok1 = pp[1] < p_hi;
            float4 sg[2]; float inv2[2]; int ivv[2]; int64_t tt[2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int64_t p = (r == 0 || ok1) ? pp[r] : pp[0];
                tt[r] = p / 5; ivv[r] = (int)(p - tt[r] * 5);
                sg[r] = __ldg(reinterpret_cast<const float4*>(&sig[tt[r]]));                // z1, z2, tha, thb
                inv2[r] = (float)(ivv[r] - 2) * 0.5f;                                       // drl_engine.py:35
            }
            // ---- TradingPolicy.forward in SGMM-F32 order (models/model.py:9-15) ----
            float h1[2][H];
#pragma unroll
            for (int j = 0; j < H; ++j) {
                const float4 w = sm.l1[j];
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    float v = __fmaf_rn(w.x, sg[r].x, w.w);
                    v = __fmaf_rn(w.y, sg[r].y, v);
                    v = __fmaf_rn(w.z, inv2[r], v);
                    h1[r][j] = fmaxf(v, 0.0f);
                }
            }
            float pa[2][H], pb[2][H];
#pragma unroll
            for (int j = 0; j < H; ++j) {
                float c0[2] = {sm.b2[j], sm.b2[j]}, c1[2] = {0.0f, 0.0f}, c2[2] = {0.0f, 0.0f}, c3[2] = {0.0f, 0.0f};
#pragma unroll
                for (int k = 0; k < H; k += 4) {
                    const float4 w = *reinterpret_cast<const float4*>(&sm.w2[j][k]);
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        c0[r] = __fmaf_rn(w.x, h1[r][k + 0], c0[r]);
                        c1[r] = __fmaf_rn(w.y, h1[r][k + 1], c1[r]);
                        c2[r] = __fmaf_rn(w.z, h1[r][k + 2], c2[r]);
                        c3[r] = __fmaf_rn(w.w, h1[r][k + 3], c3[r]);
                    }
                }
                const float2 w3 = sm.w3[j];
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    const float h2 = fmaxf(__fadd_rn(__fadd_rn(c0[r], c2[r]), __fadd_rn(c1[r], c3[r])), 0.0f);
                    pa[r][j] = __fmul_rn(w3.x, h2);
                    pb[r][j] = __fmul_rn(w3.y, h2);
                }
            }
#pragma unroll
            for (int r = 0; r < 2; ++r) {
#pragma unroll
                for (int m = 16; m >= 1; m >>= 1) {
#pragma unroll
                    for (int l = 0; l < m; ++l) { pa[r][l] = __fadd_rn(pa[r][l], pa[r][l + m]); pb[r][l] = __fadd_rn(pb[r][l], pb[r][l + m]); }
                }
                if (r == 1 && !ok1) break;
                const int64_t p = pp[r], t = tt[r];
                const int iv = ivv[r];
                const float ra = __fadd_rn(pa[r][0], sm.b3[0]), rb = __fadd_rn(pb[r][0], sm.b3[1]);
                if constexpr (RAW_OUT) { codei[p] = make_float2(ra, rb); continue; }
                const float qa = __fmul_rn(ra, 5.0f), qb = __fmul_rn(rb, 5.0f);               // raw*5.0 (drl_engine.py:39)
                if (raw) { codei[p] = make_float2(qa, qb); continue; }                        // adversary: the fills depend on the walk's state
                // ---- integer half of the env step: rounding folded into the per-bar float thresholds, as rollout_kernel_h32 ----
                const bool fb = (inv2[r] < 1.0f) && (qb < sg[r].w);                           // market_env.py:34,37
                const bool fs = (inv2[r] > -1.0f) && (qa < sg[r].z);                          // :35,:38
                codei[p] = make_float2(fs ? qa : __int_as_float(SGMM_CODE_NOFILL_F), fb ? qb : __int_as_float(SGMM_CODE_NOFILL_F));
                nexti[t * 8 + iv] = (uint8_t)(iv + (fb ? 1 : 0) - (fs ? 1 : 0));              // :45,:51
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// The walk (walk_account_kernel below) runs over one of two automata; each gives its map type, the map of bar t and the
// step of bar t from a state:
//   Walk5   no adversary: the state is the inventory index 0..4, the map of a bar comes from the table's `next` bytes.
//   Walk20  with the adversary (drl_engine.py:42-48) the walk has 20 states (fill_sell_prev, fill_buy_prev, inventory):
//           the policy table holds the raw q = raw*5 of every (bar, inventory) pair, every bar is a map {0..19} -> {0..19}
//           built from it, the bar's integer thresholds and the individual's 20-entry displacement table.
// ---------------------------------------------------------------------------------------------

struct Walk5 {
    using Map = uint32_t;
    static constexpr int STATES = 5, SCAN_UNROLL = 5;
    struct Step { float2 q; bool fb, fs; uint32_t next; };
    const float2* code;                    // this individual's [T][5] q of each side that filled, NaN marker otherwise
    const uint8_t* next;                   // [T][8] next inventory index
    template <class Pop, int OBJ>
    __device__ Walk5(const BarSig*, const float2* code_all, const uint8_t* next_all, const Pop&, int64_t ind, int64_t T,
                     std::integral_constant<int, OBJ>)
        : code(code_all + ind * T * 5), next(next_all + ind * T * 8) {}
    __device__ static Map identity() { return MAP_ID; }
    __device__ static Map then(Map f, Map g) { return map_then(f, g); }
    __device__ static Map shfl_up(Map m, int d) { return __shfl_up_sync(0xffffffffu, m, d); }
    __device__ static uint32_t at(Map m, uint32_t s) { return map_at(m, s); }
    __device__ static int inventory_index(uint32_t s) { return (int)s; }
    __device__ Map bar_map(int64_t t) const { return map_of(next + t * 8); }
    __device__ Step step(uint32_t iv, int64_t t) const
    {
        Step r;
        r.q = code[t * 5 + iv];
        r.fs = __float_as_int(r.q.x) != SGMM_CODE_NOFILL_F;
        r.fb = __float_as_int(r.q.y) != SGMM_CODE_NOFILL_F;
        r.next = next[t * 8 + iv];
        return r;
    }
    // the offsets of a bar that traded (drl_engine.py:39)
    __device__ static int2 offsets(const Step& r) { return make_int2(__float2int_rn(r.q.x), __float2int_rn(r.q.y)); }
};

struct Walk20 {
    using Map = Map20;
    static constexpr int STATES = 20, SCAN_UNROLL = 1;
    using Step = AdvStep;
    const BarSig* sig;
    const float2* code;                    // this individual's [T][5] raw q = raw*5
    uint32_t at0, at1, at2;                // displacement table (sgmm_adversary.cuh)
    // OBJ (the walk's objective) only gives each kernel its own s_adv: a table that two kernels share moves out of the
    // kernel to module scope, which shifts the shared-memory layout (and the code) of the reward kernel
    template <class Pop, int OBJ>
    __device__ Walk20(const BarSig* sig_, const float2* code_all, const uint8_t*, const Pop& adv_in, int64_t ind, int64_t T,
                      std::integral_constant<int, OBJ>)
        : sig(sig_), code(code_all + ind * T * 5)
    {
        __shared__ uint32_t s_adv[3];
        build_adv_table(adv_in, ind, s_adv);
        at0 = s_adv[0]; at1 = s_adv[1]; at2 = s_adv[2];
    }
    __device__ static Map identity() { return m20_identity(); }
    __device__ static Map then(const Map& f, const Map& g) { return m20_then(f, g); }
    __device__ static Map shfl_up(const Map& m, int d) { return m20_shfl_up(m, d); }
    __device__ static uint32_t at(const Map& m, uint32_t s) { return m20_at(m, s); }
    __device__ static int inventory_index(uint32_t s) { return (int)(s % 5u); }
    __device__ int2 k1(int64_t t) const { return __ldg(reinterpret_cast<const int2*>(&sig[t].ka1)); }
    __device__ Map bar_map(int64_t t) const
    {
        Map20 m = {{0u, 0u, 0u, 0u}};
        bar_map_rec(m, code + t * 5, k1(t), at0, at1, at2);
        return m;
    }
    __device__ Step step(uint32_t st, int64_t t) const { return adv_step(st, code + t * 5, k1(t), at0, at1, at2); }
    __device__ static int2 offsets(const Step& r) { return make_int2(r.oa, r.ob); }
};

// phi and fee of this CTA's episode: the launch's (a population), or those of its individual's run (a GA sweep)
__device__ __forceinline__ double cta_phi(const PopArgs&, double phi) { return phi; }
__device__ __forceinline__ double cta_fee(const PopArgs&, double fee) { return fee; }
__device__ __forceinline__ const GaDev* cta_run(const SweepPop& p) { return p.st + (p.first + (int64_t)blockIdx.x) / p.lambda; }
__device__ __forceinline__ double cta_phi(const SweepPop& p, double) { return cta_run(p)->phi; }
__device__ __forceinline__ double cta_fee(const SweepPop& p, double) { return cta_run(p)->fee; }

// CTAs per SM of the 512-thread walk without the adversary: 3 (40 registers); a sweep's CTA also keeps its run's phi / fee
// and takes 2, so that it runs in 64 registers without spilling
template <class Pop> constexpr int walk_ctas_per_sm() { return 3; }
template <> constexpr int walk_ctas_per_sm<SweepPop>() { return 2; }

// Phase 3 of walk_account_kernel for a StrategyAnalytics objective (sgmm.h, SGMM_OBJECTIVE_*), chunk by chunk of OBJ_CHUNK
// bars: every thread steps its own bars and stages the two cash terms (my_bid + fee, my_ask - fee) in s_buf (both halves
// of the reward kernel's s_rew), the fill bits and the inventory after the bar; one thread runs the cash chain in bar
// order (buy leg, then sell leg, as env_step); then wealth = cash + inventory * mid_next in parallel, the expression of
// sgmm_trace_pop.cu.  Total PnL needs the first and last wealth, MAP the sum of |inventory| (an integer: any order), the
// Sharpe the wealth differences of consecutive trade rows, which one thread appends in bar order to `scratch` before the
// two pairwise passes of analytics_kernel (trade_sharpe).  Every thread of the CTA calls it.
constexpr int OBJ_CHUNK = SUM_CHUNK / 2;

template <class A, int WALK_THREADS, int OBJ>
__device__ __forceinline__ void walk_objective(const A& w, uint32_t st, int64_t t_lo, int64_t t_hi, int64_t T,
                                               const BarPx* __restrict__ px, double tick, double fee, double* s_buf,
                                               int* s_trades, double* __restrict__ obj_scratch, double* __restrict__ fitness,
                                               int32_t* __restrict__ trades)
{
    __shared__ uint8_t s_out[OBJ_CHUNK];                    // fill_buy | fill_sell << 1 | inventory index after the bar << 2
    __shared__ unsigned long long s_abs;
    __shared__ double s_w0, s_wl;
    double* s_cb = s_buf;                                   // cash term of the buy leg, then the cash after the bar
    double* s_cs = s_buf + OBJ_CHUNK;                       // cash term of the sell leg, then (SHARPE) the wealth
    const int tid = threadIdx.x;
    if (tid == 0) { s_abs = 0ull; s_w0 = 0.0; s_wl = 0.0; }
    double* scratch = OBJ == SGMM_OBJECTIVE_SHARPE ? obj_scratch + (int64_t)blockIdx.x * T : nullptr;
    int ntr = 0, abs_inv = 0;
    double cash = 0.0, prev = 0.0;                          // thread 0: the cash chain, the last trade row's wealth
    int64_t m = 0;                                          // thread 0: wealth differences written
    bool seen = false;                                      // thread 0: a trade row has been met
    for (int64_t c0 = 0; c0 < T; c0 += OBJ_CHUNK) {
        const int64_t c1 = c0 + OBJ_CHUNK < T ? c0 + OBJ_CHUNK : T;
        const int n = (int)(c1 - c0);
        const int64_t a = t_lo > c0 ? t_lo : c0, b = t_hi < c1 ? t_hi : c1;
        for (int64_t t = a; t < b; ++t) {
            const typename A::Step r = w.step(st, t);
            const int iv = A::inventory_index(r.next);
            ntr += (r.fb || r.fs) ? 1 : 0;                                         // drl_engine.py:60-61
            abs_inv += iv > 2 ? iv - 2 : 2 - iv;                                   // mm_analyzer.py:27
            double cb = 0.0, cs = 0.0;
            if (r.fb || r.fs) {
                const BarPx p = px[t];
                const int2 k = A::offsets(r);
                const double my_ask = quote_ask(p.ask, k.x, tick), my_bid = quote_bid(p.bid, k.y, tick);     // market_env.py:30-31
                cb = add_rn(my_bid, mul_rn(my_bid, fee));                                                    // :47
                cs = sub_rn(my_ask, mul_rn(my_ask, fee));                                                    // :53
            }
            s_cb[t - c0] = cb; s_cs[t - c0] = cs;
            s_out[t - c0] = (uint8_t)((r.fb ? 1 : 0) | (r.fs ? 2 : 0) | (iv << 2));
            st = r.next;
        }
        __syncthreads();
        if (tid == 0) {
            for (int i = 0; i < n; ++i) {
                const int f = s_out[i];
                if (f & 1) cash = sub_rn(cash, s_cb[i]);
                if (f & 2) cash = add_rn(cash, s_cs[i]);
                s_cb[i] = cash;
            }
        }
        __syncthreads();
        for (int i = tid; i < n; i += WALK_THREADS) {
            const int64_t t = c0 + i;
            if (OBJ == SGMM_OBJECTIVE_SHARPE || t == 0 || t == T - 1) {
                const double wl = add_rn(s_cb[i], mul_rn((double)((s_out[i] >> 2) - 2), px[t].mid_next));   // Env/recorder.py:46
                if (t == 0) s_w0 = wl;
                if (t == T - 1) s_wl = wl;
                if (OBJ == SGMM_OBJECTIVE_SHARPE) s_cs[i] = wl;
            }
        }
        if constexpr (OBJ == SGMM_OBJECTIVE_SHARPE) {
            __syncthreads();
            if (tid == 0) {
                for (int i = 0; i < n; ++i) {
                    if (s_out[i] & 3) {                                            // mm_analyzer.py:10,39
                        const double wl = s_cs[i];
                        if (seen) scratch[m++] = sub_rn(wl, prev);
                        prev = wl; seen = true;
                    }
                }
            }
        }
        __syncthreads();
    }
    if (ntr) atomicAdd(s_trades, ntr);
    if (abs_inv) atomicAdd(&s_abs, (unsigned long long)abs_inv);
    __syncthreads();
    if (tid == 0) {
        const int nt = *s_trades;
        const double total = sub_rn(s_wl, s_w0);                                   // mm_analyzer.py:15
        double v;
        if constexpr (OBJ == SGMM_OBJECTIVE_PNL) v = total;
        else if constexpr (OBJ == SGMM_OBJECTIVE_PNL_MAP) {
            const double map = T > 0 ? __ddiv_rn((double)s_abs, (double)T) : 0.0;    // :27
            v = map == 0.0 ? 0.0 : __ddiv_rn(total, map);
        } else v = trade_sharpe(scratch, m, nt);
        fitness[blockIdx.x] = objective_fitness(v, nt); trades[blockIdx.x] = nt;
    }
}

// One CTA per individual.  WALK_THREADS = 1024 (one individual per SM: shortest latency, populations up to the SM count) or
// 512 (three per SM without the adversary: the serial reward sum of one individual hides behind the others).
// Pop: PopArgs (phi_arg / fee_arg apply to every CTA), or SweepPop (a GA sweep: CTA i walks individual adv.first + i of the
// sweep with its run's phi and fee; with the adversary, adv gives the individual's seeded adversary).
// OBJ: the training objective (SGMM_OBJECTIVE_*).  REWARD sums the reference's rewards; the others run the cash chain
// instead and reduce wealth to the StrategyAnalytics column (phase 3 below).  SHARPE writes the wealth differences of
// consecutive trade rows of CTA i to obj_scratch[i][0 .. trades-1) (T doubles per CTA).  An objective CTA keeps the cash
// chain, the first and last wealth and the Sharpe state in registers: two CTAs per SM at 512 threads, 64 registers.
template <class A, int WALK_THREADS, class Pop, int OBJ = SGMM_OBJECTIVE_REWARD>
__global__ void __launch_bounds__(WALK_THREADS, (WALK_THREADS == 1024 || A::STATES == 20) ? 1 : (OBJ != SGMM_OBJECTIVE_REWARD ? 2 : walk_ctas_per_sm<Pop>()))
walk_account_kernel(const BarSig* __restrict__ sig, const BarPx* __restrict__ px, int64_t T, const float2* __restrict__ code_all,
                    const uint8_t* __restrict__ next_all, const Pop adv, double tick, double phi_arg, double fee_arg,
                    double* __restrict__ fitness, int32_t* __restrict__ trades, double* __restrict__ obj_scratch)
{
    using Map = typename A::Map;
    __shared__ Map s_warp[32];                              // (WALK_THREADS / 32 entries used)
    __shared__ int s_trades;
    __shared__ double s_rew[SUM_CHUNK];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_trades = 0;
    const A w(sig, code_all, next_all, adv, blockIdx.x, T, std::integral_constant<int, OBJ>{});
    // ---- 1. every thread composes the maps of its contiguous segment of bars ----
    const int64_t L = (T + WALK_THREADS - 1) / WALK_THREADS;
    const int64_t t_lo = (int64_t)tid * L < T ? (int64_t)tid * L : T, t_hi = t_lo + L < T ? t_lo + L : T;
    Map m = A::identity();
    for (int64_t t = t_lo; t < t_hi; ++t) m = A::then(m, w.bar_map(t));
    // ---- 2. exclusive scan over the segments (composition is associative, not commutative: earlier bars first) ----
    Map inc = m;
#pragma unroll A::SCAN_UNROLL
    for (int d = 1; d < 32; d <<= 1) {
        const Map o = A::shfl_up(inc, d);
        if (lane >= d) inc = A::then(o, inc);
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        Map v = lane < WALK_THREADS / 32 ? s_warp[lane] : A::identity();
#pragma unroll A::SCAN_UNROLL
        for (int d = 1; d < 32; d <<= 1) {
            const Map o = A::shfl_up(v, d);
            if (lane >= d) v = A::then(o, v);
        }
        s_warp[lane] = v;                                   // inclusive over warps
    }
    __syncthreads();
    Map before = A::shfl_up(inc, 1);                        // everything before this thread inside its warp
    if (lane == 0) before = A::identity();
    if (warp > 0) before = A::then(s_warp[warp - 1], before);
    uint32_t st = A::at(before, 2u);                        // flat, no previous fills: state 2 (market_env.py:17, drl_engine.py:29)
    if constexpr (OBJ != SGMM_OBJECTIVE_REWARD) {
        walk_objective<A, WALK_THREADS, OBJ>(w, st, t_lo, t_hi, T, px, tick, cta_fee(adv, fee_arg), s_rew, &s_trades,
                                             obj_scratch, fitness, trades);
        return;
    }
    // ---- 3. the fp64 half for the visited states, chunk by chunk; one thread sums each chunk in bar order ----
    const PenaltyTable pen = penalty_table(cta_phi(adv, phi_arg));
    int ntr = 0;
    double total = 0.0;                                     // thread 0 only (drl_engine.py:26)
    for (int64_t c0 = 0; c0 < T; c0 += SUM_CHUNK) {
        const int64_t c1 = c0 + SUM_CHUNK < T ? c0 + SUM_CHUNK : T;
        const int64_t a = t_lo > c0 ? t_lo : c0, b = t_hi < c1 ? t_hi : c1;       // this thread's bars inside the chunk
        for (int64_t t = a; t < b; ++t) {
            const typename A::Step r = w.step(st, t);
            ntr += (r.fb || r.fs) ? 1 : 0;                                         // drl_engine.py:60-61
            double pnl = 0.0;                                                      // market_env.py:40
            if (r.fb || r.fs) {
                const BarPx p = px[t];
                const int2 k = A::offsets(r);
                const double my_ask = quote_ask(p.ask, k.x, tick), my_bid = quote_bid(p.bid, k.y, tick);         // :30-31
                // fee terms evaluated as the reference does, fee_rate 0 included
                const double fee = cta_fee(adv, fee_arg);
                const double leg_b = buy_leg(my_bid, p.mid_next, fee), leg_s = sell_leg(my_ask, p.mid_next, fee);
                pnl = r.fb ? add_rn(pnl, leg_b) : pnl;
                pnl = r.fs ? add_rn(pnl, leg_s) : pnl;
            }
            s_rew[t - c0] = sub_rn(pnl, penalty(pen, abs(A::inventory_index(r.next) - 2)));      // :57-58
            st = r.next;
        }
        __syncthreads();
        if (tid == 0) {
            const int n = (int)(c1 - c0);
            for (int i = 0; i < n; ++i) total = add_rn(total, s_rew[i]);           // drl_engine.py:54
        }
        __syncthreads();
    }
    if (ntr) atomicAdd(&s_trades, ntr);
    __syncthreads();
    if (tid == 0) {
        const int n = s_trades;
        fitness[blockIdx.x] = episode_fitness(total, n); trades[blockIdx.x] = n;
    }
}

// Audit of a walk over q tables: the market maker's offsets before the displacement at the state walk_account_kernel<Walk20>
// visits, bar after bar on one thread (the offsets tests replay through the oracle; not a hot path).  One CTA per individual.
__global__ void __launch_bounds__(32) adv_offsets_kernel(const BarSig* __restrict__ sig, int64_t T, const float2* __restrict__ code_all,
                                                         const PopArgs adv, int32_t* __restrict__ act_trace)
{
    __shared__ uint32_t s_adv[3];                           // its own: sharing Walk20's static table would move walk_account_kernel's shared layout
    build_adv_table(adv, blockIdx.x, s_adv);
    if (threadIdx.x != 0) return;
    const float2* code = code_all + (int64_t)blockIdx.x * T * 5;
    int32_t* act = act_trace + (int64_t)blockIdx.x * T * 2;
    uint32_t st = 2u;                                       // flat, no previous fills
    for (int64_t t = 0; t < T; ++t) {
        const float2 q = code[t * 5 + st % 5u];
        act[2 * t] = mm_offset(q.x); act[2 * t + 1] = mm_offset(q.y);
        st = adv_step(st, code + t * 5, __ldg(reinterpret_cast<const int2*>(&sig[t].ka1)), s_adv[0], s_adv[1], s_adv[2]).next;
    }
}

}  // namespace one

namespace one {
// grid and pairs per task of policy_table_kernel for P individuals: task = (individual, range of pairs), ranges of whole
// 128-pair rounds, sized so that the GPU gets ~8 blocks per SM
static unsigned policy_table_grid(const sgmm_bundle* b, int64_t P, bool seeded, int64_t* pairs_per_task)
{
    const int64_t T = b->T;
    const int64_t want_blocks = (int64_t)sm_count(b->device) * 8;
    int64_t ppt = (P * T * 5 + want_blocks - 1) / want_blocks;
    ppt = (ppt + 2 * PT_THREADS - 1) / (2 * PT_THREADS) * (2 * PT_THREADS);
    const int64_t ppt_min = seeded ? 4 * PT_THREADS : 2 * PT_THREADS;          // seeded children: staging costs ~10 Philox calls per thread
    if (ppt < ppt_min) ppt = ppt_min;
    const int64_t ntasks = P * ((T * 5 + ppt - 1) / ppt);
    const int64_t blocks = ntasks < want_blocks * 2 ? ntasks : want_blocks * 2;
    *pairs_per_task = ppt;
    return (unsigned)(blocks < 1 ? 1 : blocks);
}

static bool seeded(const PopArgs& p) { return p.genomes == nullptr; }
static bool seeded(const SweepPop&) { return true; }

// the table callback of table_walk_batches on this path: step codes + next inventory, or q tables with the adversary
inline auto policy_tables(const sgmm_bundle* b, cudaStream_t st)
{
    return [b, st](const auto& pm, const auto* pa, int64_t, const BatchScratch& s) {
        return launch_policy_table(b, pm, pa ? 1 : 0, s.code, s.next, st);
    };
}
}  // namespace one

template <class Pop>
int launch_policy_table(const sgmm_bundle* b, const Pop& mm, int mode, float2* code, uint8_t* next, cudaStream_t st)
{
    using namespace one;
    const int64_t T = b->T, P = mm.count;
    if (T == 0 || P == 0) return SGMM_OK;
    int64_t ppt = 0;
    const unsigned grid = policy_table_grid(b, P, seeded(mm), &ppt);
    if constexpr (std::is_same<Pop, PopArgs>::value)          // raw outputs: the population trace (no sweep instantiation)
        if (mode == 2) {
            policy_table_kernel<true><<<grid, PT_THREADS, 0, st>>>(b->sig, T, mm, ppt, 0, code, next);
            return check_cuda(cudaGetLastError(), "policy_table_kernel launch");
        }
    policy_table_kernel<false><<<grid, PT_THREADS, 0, st>>>(b->sig, T, mm, ppt, mode, code, next);
    return check_cuda(cudaGetLastError(), "policy_table_kernel launch");
}

namespace one {
template <int OBJ, class Pop>
static void launch_walk_as(const sgmm_bundle* b, int64_t P, const float2* code, const uint8_t* next, const Pop& pop, bool adv,
                           double phi, double fee, double* fitness, int32_t* trades, double* obj_scratch, cudaStream_t st)
{
    const int64_t T = b->T;
    if (adv) walk_account_kernel<Walk20, 512, Pop, OBJ><<<(unsigned)P, 512, 0, st>>>(b->sig, b->px, T, code, nullptr, pop, b->tick, phi, fee, fitness, trades, obj_scratch);
    else if (P <= sm_count(b->device)) walk_account_kernel<Walk5, 1024, Pop, OBJ><<<(unsigned)P, 1024, 0, st>>>(b->sig, b->px, T, code, next, pop, b->tick, phi, fee, fitness, trades, obj_scratch);
    else walk_account_kernel<Walk5, 512, Pop, OBJ><<<(unsigned)P, 512, 0, st>>>(b->sig, b->px, T, code, next, pop, b->tick, phi, fee, fitness, trades, obj_scratch);
}
}  // namespace one

template <class Pop>
int launch_walk(const sgmm_bundle* b, int64_t P, const float2* code, const uint8_t* next, const Pop& pop, bool adv, double phi,
                double fee, double* fitness, int32_t* trades, int objective, double* obj_scratch, cudaStream_t st)
{
    using namespace one;
    switch (objective) {
        case SGMM_OBJECTIVE_PNL: launch_walk_as<SGMM_OBJECTIVE_PNL>(b, P, code, next, pop, adv, phi, fee, fitness, trades, obj_scratch, st); break;
        case SGMM_OBJECTIVE_PNL_MAP: launch_walk_as<SGMM_OBJECTIVE_PNL_MAP>(b, P, code, next, pop, adv, phi, fee, fitness, trades, obj_scratch, st); break;
        case SGMM_OBJECTIVE_SHARPE: launch_walk_as<SGMM_OBJECTIVE_SHARPE>(b, P, code, next, pop, adv, phi, fee, fitness, trades, obj_scratch, st); break;
        default: launch_walk_as<SGMM_OBJECTIVE_REWARD>(b, P, code, next, pop, adv, phi, fee, fitness, trades, obj_scratch, st); break;
    }
    return check_cuda(cudaGetLastError(), "walk_account_kernel launch");
}

template int launch_policy_table<PopArgs>(const sgmm_bundle*, const PopArgs&, int, float2*, uint8_t*, cudaStream_t);
template int launch_policy_table<SweepPop>(const sgmm_bundle*, const SweepPop&, int, float2*, uint8_t*, cudaStream_t);
template int launch_walk<PopArgs>(const sgmm_bundle*, int64_t, const float2*, const uint8_t*, const PopArgs&, bool, double, double,
                                  double*, int32_t*, int, double*, cudaStream_t);
template int launch_walk<SweepPop>(const sgmm_bundle*, int64_t, const float2*, const uint8_t*, const SweepPop&, bool, double, double,
                                   double*, int32_t*, int, double*, cudaStream_t);

// Episodes of a small population on `b` (H = 32, exact SGMM-F32 order, with or without the adversary) through the kernels
// above.  The policy table ([count][T] x 48 B) lives in the bundle's code buffer, as batches of table_walk_batches: one
// batch at the default budget.  A non-REWARD objective takes this route at every population size.
int launch_rollout_small(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, double phi, double fee, double* fitness, int32_t* trades,
                         cudaStream_t st, int objective)
{
    return table_walk_batches(b, mm, adv, mm, genome_len(32), true, 0, phi, fee, fitness, trades, st, one::policy_tables(b, st), objective);
}

// The K*lambda children of a GA sweep take the policy-table path whatever their number (a solo GA of more than
// SMALL_POP_MAX children runs rollout_kernel_h32, which gives the same bits).  The table ([n][T] x 48 B) lives in the
// bundle's code buffer, in batches of n individuals; a batch may start inside a run.  phi / fee are the runs'.
int launch_sweep_population(const sgmm_bundle* b, const SweepPop& mm, const SweepPop* adv, double* fitness, int32_t* trades,
                            cudaStream_t st, int objective)
{
    return table_walk_batches(b, mm, adv, mm, genome_len(32), true, 0, 0.0, 0.0, fitness, trades, st, one::policy_tables(b, st),
                              objective);
}

// The K masters of a sweep, contiguous [K][1250] rows, as one explicit population (adversary off, as the validation of a
// solo GA); the walk's CTA r takes run r's phi and fee
int launch_sweep_validation(const sgmm_bundle* b, const float* masters, const GaDev* runs, int64_t K, double* fitness,
                            int32_t* trades, cudaStream_t st, int objective)
{
    PopArgs pm{};
    pm.genomes = masters; pm.count = K;
    const SweepPop all{nullptr, runs, 1, 0, K, 0};
    return table_walk_batches(b, pm, (const PopArgs*)nullptr, all, genome_len(32), true, 0, 0.0, 0.0, fitness, trades, st,
                              one::policy_tables(b, st), objective);
}

int launch_adv_offsets(const sgmm_bundle* b, int64_t P, const float2* code, const PopArgs& adv, int32_t* act_trace, cudaStream_t st)
{
    if (P == 0) return SGMM_OK;
    one::adv_offsets_kernel<<<(unsigned)P, 32, 0, st>>>(b->sig, b->T, code, adv, act_trace);
    return check_cuda(cudaGetLastError(), "adv_offsets_kernel launch");
}

}  // namespace sgmm
