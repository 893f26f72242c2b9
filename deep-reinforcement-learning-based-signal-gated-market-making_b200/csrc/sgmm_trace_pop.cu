// sgmm_trace_pop.cu -- recorder traces of a whole population in one call (sgmm_rollout_trace_population): every column of
// sgmm_trace for every individual, row i bit-identical to sgmm_rollout_trace of individual i alone (trace_kernel_h32, which
// walks the bars of one individual on one warp).
//
//   1. the raw policy outputs (before x5) of every (bar, inventory) pair, float2 [n][T][5], in SGMM-F32 order:
//      one::policy_table_kernel<true> at H = 32, x256::exact256_table_kernel mode 2 at H = 256;
//   2. trace_pop_kernel, one CTA per individual:
//      a. the walk of walk_account_kernel -- maps of the thread segments composed, exclusive scan over the block -- over the
//         5-state automaton (the 20-state one with the adversary) built from q = fl(raw*5) and the bar's thresholds: the
//         state entering every thread's first bar;
//      b. per chunk of CHUNK bars, every thread steps its own bars inside the chunk and records the state entering each;
//         then the chunk's bars in parallel, consecutive bars on consecutive threads (coalesced writes): offsets,
//         displacement, the literal env_step on the raw bounds from the entering inventory, the per-bar columns, and the
//         terms of the three serial fp64 chains, staged in shared memory;
//      c. three threads in different warps run the chains in bar order over the chunk -- cash (buy leg, then sell leg, as
//         env_step applies them), the reward sum (its last value, through episode_fitness, is the fitness) and the fee sum
//         -- and the block writes cash, wealth, cum_reward and cum_fees back.
// A NULL column is not written, and the work only it needs is skipped (the cash chain without cash and wealth, the fee
// chain without cum_fees).
#include "sgmm_internal.h"
#include "sgmm_step_core.h"
#include "sgmm_walk.cuh"

namespace sgmm {

namespace tpop {

constexpr int THREADS = 256;
constexpr int CHUNK = 2048;                // bars whose chain terms sit in shared memory at a time

struct Smem {
    double cb[CHUNK];                      // cash term of the buy leg (my_bid + fee), then cash after the bar
    double cs[CHUNK];                      // cash term of the sell leg (my_ask - fee)
    double rew[CHUNK];                     // reward, then its running sum
    double fee[CHUNK];                     // fee_paid, then its running sum
    uint8_t st[CHUNK];                     // state entering the bar
    uint8_t out[CHUNK];                    // fill_buy | fill_sell << 1 | (inventory after the bar + 2) << 2
};

struct Args {
    const BarSig* sig; const BarPx* px; const double* bmax; const double* smin;
    int64_t T; double tick, phi, fee;
    const float2* raw;                     // [n][T][5] raw policy outputs
    PopArgs adv;                           // the batch's adversaries (count 0: none)
    sgmm_trace tr;                         // columns of the batch's first row
    double* fitness; int32_t* trades;
};

__device__ __forceinline__ float2 q_of(float2 r) { return make_float2(__fmul_rn(r.x, 5.0f), __fmul_rn(r.y, 5.0f)); }   // drl_engine.py:39

// no adversary: the state is the inventory index; fills from q against the bar's float thresholds, as policy_table_kernel
struct RawWalk5 {
    using Map = uint32_t;
    static constexpr int STATES = 5, SCAN_UNROLL = 5;
    const BarSig* sig;
    const float2* raw;                     // this individual's [T][5]
    uint32_t at0, at1, at2;                // (unused)
    __device__ static Map identity() { return one::MAP_ID; }
    __device__ static Map then(Map f, Map g) { return one::map_then(f, g); }
    __device__ static Map shfl_up(Map m, int d) { return __shfl_up_sync(0xffffffffu, m, d); }
    __device__ static uint32_t at(Map m, uint32_t s) { return one::map_at(m, s); }
    __device__ static int inventory_index(uint32_t s) { return (int)s; }
    __device__ static uint32_t next_of(uint32_t iv, float2 q, float4 s)
    {
        const bool fb = (iv < 4u) && (q.y < s.w);                                          // market_env.py:34,37
        const bool fs = (iv > 0u) && (q.x < s.z);                                          // :35,:38
        return iv + (fb ? 1u : 0u) - (fs ? 1u : 0u);
    }
    __device__ Map bar_map(int64_t t) const
    {
        const float4 s = __ldg(reinterpret_cast<const float4*>(&sig[t]));
        Map m = 0;
#pragma unroll
        for (uint32_t iv = 0; iv < 5u; ++iv) m |= next_of(iv, q_of(raw[t * 5 + iv]), s) << (3u * iv);
        return m;
    }
    __device__ uint32_t step(uint32_t st, int64_t t) const
    {
        return next_of(st, q_of(raw[t * 5 + st]), __ldg(reinterpret_cast<const float4*>(&sig[t])));
    }
};

// with the adversary: the 20-state automaton of walk_account_kernel<Walk20>
struct RawWalk20 {
    using Map = one::Map20;
    static constexpr int STATES = 20, SCAN_UNROLL = 1;
    const BarSig* sig;
    const float2* raw;
    uint32_t at0, at1, at2;                // displacement table (sgmm_adversary.cuh)
    __device__ static Map identity() { return one::m20_identity(); }
    __device__ static Map then(const Map& f, const Map& g) { return one::m20_then(f, g); }
    __device__ static Map shfl_up(const Map& m, int d) { return one::m20_shfl_up(m, d); }
    __device__ static uint32_t at(const Map& m, uint32_t s) { return one::m20_at(m, s); }
    __device__ static int inventory_index(uint32_t s) { return (int)(s % 5u); }
    __device__ int2 k1(int64_t t) const { return __ldg(reinterpret_cast<const int2*>(&sig[t].ka1)); }
    __device__ Map bar_map(int64_t t) const
    {
        float2 q[5];
#pragma unroll
        for (int iv = 0; iv < 5; ++iv) q[iv] = q_of(raw[t * 5 + iv]);
        Map m = {{0u, 0u, 0u, 0u}};
        one::bar_map_rec(m, q, k1(t), at0, at1, at2);
        return m;
    }
    __device__ uint32_t step(uint32_t st, int64_t t) const
    {
        return one::adv_step_q(st, q_of(raw[t * 5 + st % 5u]), k1(t), at0, at1, at2).next;
    }
};

// The state entering the first bar of this thread's segment, m being the composition of the segment's bar maps: an exclusive
// scan over the block's segments (composition is associative, not commutative: earlier bars first) applied to the first
// state 2 (flat, no previous fills: market_env.py:17, drl_engine.py:29).  s_warp: 32 maps of shared memory; every thread of
// the block calls it.  The same scan as walk_account_kernel's, which keeps its own inline copy: called through this function
// it allocates registers differently.
template <class A, int WALK_THREADS>
__device__ __forceinline__ uint32_t entering_state(typename A::Map m, typename A::Map* s_warp)
{
    using Map = typename A::Map;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
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
    return A::at(before, 2u);
}

template <class A>
__global__ void __launch_bounds__(THREADS, 2) trace_pop_kernel(const Args a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    using Map = typename A::Map;
    __shared__ Map s_warp[32];
    __shared__ uint32_t s_adv[3];
    __shared__ int s_trades;
    const int tid = threadIdx.x;
    const int64_t T = a.T, ind = blockIdx.x;
    if (tid == 0) s_trades = 0;
    A w;
    w.sig = a.sig; w.raw = a.raw + ind * T * 5;
    w.at0 = w.at1 = w.at2 = 0u;
    constexpr bool ADV = A::STATES == 20;
    if constexpr (ADV) {
        one::build_adv_table(a.adv, ind, s_adv);
        w.at0 = s_adv[0]; w.at1 = s_adv[1]; w.at2 = s_adv[2];
    }
    // ---- a. the walk: the state entering this thread's segment ----
    const int64_t L = (T + THREADS - 1) / THREADS;
    const int64_t t_lo = (int64_t)tid * L < T ? (int64_t)tid * L : T, t_hi = t_lo + L < T ? t_lo + L : T;
    Map m = A::identity();
    for (int64_t t = t_lo; t < t_hi; ++t) m = A::then(m, w.bar_map(t));
    uint32_t st = entering_state<A, THREADS>(m, s_warp);

    const sgmm_trace& tr = a.tr;
    const bool need_cash = tr.cash || tr.wealth, need_fees = tr.cum_fees != nullptr;
    const int64_t row = ind * T;
    int ntr = 0;
    double chain = 0.0;                    // thread 0: cash, thread 32: the reward sum, thread 64: the fee sum
    for (int64_t c0 = 0; c0 < T; c0 += CHUNK) {
        const int64_t c1 = c0 + CHUNK < T ? c0 + CHUNK : T;
        const int n = (int)(c1 - c0);
        // ---- b. the states entering this thread's bars of the chunk, then every bar of the chunk in parallel ----
        for (int64_t t = t_lo > c0 ? t_lo : c0, e = t_hi < c1 ? t_hi : c1; t < e; ++t) {
            sm.st[t - c0] = (uint8_t)st;
            st = w.step(st, t);
        }
        __syncthreads();
        for (int i = tid; i < n; i += THREADS) {
            const int64_t t = c0 + i, o = row + t;
            const uint32_t s = sm.st[i];
            const int iv = A::inventory_index(s);
            const float2 r = w.raw[t * 5 + iv];
            const int ka = __float2int_rn(__fmul_rn(r.x, 5.0f)), kb = __float2int_rn(__fmul_rn(r.y, 5.0f));   // drl_engine.py:39
            int da = 0, db = 0;
            if constexpr (ADV) {
                const uint32_t e = table_lookup(w.at0, w.at1, w.at2, (int)s);
                da = (int)(e & 3u) - 1; db = (int)(e >> 2) - 1;                            // market_env.py:26-28
            }
            const BarPx px = a.px[t];
            sgmm_env_state env;
            env.phi = a.phi; env.tick_size = a.tick; env.fee_rate = a.fee;
            env.inventory = iv - 2; env.cash = 0.0; env.i_max = 2; env.i_min = -2;
            const int64_t oa = (int64_t)ka + da, ob = (int64_t)kb + db;
            sgmm_step_info info;
            env_step(env, oa, ob, px.mid_next, px.ask, px.bid, a.bmax[t], a.smin[t], info);
            ntr += info.fill_buy | info.fill_sell;
            if (tr.off_a) tr.off_a[o] = ka;
            if (tr.off_b) tr.off_b[o] = kb;
            if (tr.adv_a) tr.adv_a[o] = da;
            if (tr.adv_b) tr.adv_b[o] = db;
            if (tr.fill_buy) tr.fill_buy[o] = info.fill_buy;
            if (tr.fill_sell) tr.fill_sell[o] = info.fill_sell;
            if (tr.inventory) tr.inventory[o] = (int32_t)env.inventory;
            if (tr.reward) tr.reward[o] = info.reward;
            if (tr.pnl_reward) tr.pnl_reward[o] = info.pnl_reward;
            if (tr.inventory_reward) tr.inventory_reward[o] = info.inventory_reward;
            if (tr.fee_paid) tr.fee_paid[o] = info.fee_paid;
            if (tr.raw_a) tr.raw_a[o] = r.x;
            if (tr.raw_b) tr.raw_b[o] = r.y;
            if (tr.spread) tr.spread[o] = sub_rn(px.ask, px.bid);
            if (tr.skew) tr.skew[o] = kb - ka;
            if (tr.unrealized_pnl) tr.unrealized_pnl[o] = mul_rn((double)env.inventory, px.mid_next);
            if (need_cash) {                                                               // market_env.py:47,53
                const double my_bid = quote_bid(px.bid, ob, a.tick), my_ask = quote_ask(px.ask, oa, a.tick);
                sm.cb[i] = add_rn(my_bid, mul_rn(my_bid, a.fee));
                sm.cs[i] = sub_rn(my_ask, mul_rn(my_ask, a.fee));
            }
            sm.rew[i] = info.reward;
            if (need_fees) sm.fee[i] = info.fee_paid;
            sm.out[i] = (uint8_t)(info.fill_buy | (info.fill_sell << 1) | ((int)(env.inventory + 2) << 2));
        }
        __syncthreads();
        // ---- c. the three fp64 chains in bar order ----
        if (tid == 0 && need_cash) {
            for (int i = 0; i < n; ++i) {
                const int f = sm.out[i];
                if (f & 1) chain = sub_rn(chain, sm.cb[i]);
                if (f & 2) chain = add_rn(chain, sm.cs[i]);
                sm.cb[i] = chain;
            }
        } else if (tid == 32) {
            for (int i = 0; i < n; ++i) { chain = add_rn(chain, sm.rew[i]); sm.rew[i] = chain; }    // drl_engine.py:54
        } else if (tid == 64 && need_fees) {
            for (int i = 0; i < n; ++i) { chain = add_rn(chain, sm.fee[i]); sm.fee[i] = chain; }    // Env/recorder.py:49
        }
        __syncthreads();
        for (int i = tid; i < n; i += THREADS) {
            const int64_t o = row + c0 + i;
            if (tr.cash) tr.cash[o] = sm.cb[i];
            if (tr.wealth) tr.wealth[o] = add_rn(sm.cb[i], mul_rn((double)((sm.out[i] >> 2) - 2), a.px[c0 + i].mid_next));   // :46
            if (tr.cum_reward) tr.cum_reward[o] = sm.rew[i];
            if (tr.cum_fees) tr.cum_fees[o] = sm.fee[i];
        }
        __syncthreads();
    }
    if (ntr) atomicAdd(&s_trades, ntr);
    __syncthreads();
    if (tid == 32) {
        const int nt = s_trades;
        a.fitness[ind] = episode_fitness(chain, nt); a.trades[ind] = nt;
    }
}

template <class A>
int launch_kernel(const Args& args, int64_t n, cudaStream_t st)
{
    static std::atomic<uint64_t> configured{0};
    if (int rc = opt_in_smem(trace_pop_kernel<A>, sizeof(Smem), configured, "cudaFuncSetAttribute(trace_pop smem)")) return rc;
    trace_pop_kernel<A><<<(unsigned)n, THREADS, sizeof(Smem), st>>>(args);
    return check_cuda(cudaGetLastError(), "trace_pop_kernel launch");
}

}  // namespace tpop

// Traces of mm.count individuals, in batches under the byte budget of x256::batch_bytes(): the raw table ([n][T] x 40 B, plus
// the staged genomes at H = 256 when seeded or unaligned) lives in the bundle's code buffer (rollouts sharing it are ordered
// across streams; the first call of a size allocates and must not run under a stream capture).  Batch b0 writes rows b0 ...
// of the caller's columns.
int launch_trace_population(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, int hidden, double phi, double fee,
                            const sgmm_trace* tr, double* fitness, int32_t* trades, cudaStream_t st)
{
    const int64_t T = b->T, P = mm.count, G = genome_len(hidden);
    if (P == 0) return SGMM_OK;
    const bool stage = hidden == 256 && T > 0 && x256::needs_stage(mm);
    int64_t nb = 0;
    uint64_t* buf = nullptr;
    if (int rc = reserve_batches(b, P, 5 * T + (stage ? G / 2 : 0), st, &nb, &buf)) return rc;
    CodesRelease release(b, st);
    float2* raw = reinterpret_cast<float2*>(buf);
    float* staged = reinterpret_cast<float*>(buf + nb * T * 5);
    sgmm_trace none = {};
    const sgmm_trace cols = tr ? *tr : none;
    const int rc = for_each_batch(mm, adv, nb, G, [&](const PopArgs& pm, const PopArgs* pa, int64_t b0) {
        if (hidden == 32) {
            if (int rc = launch_policy_table(b, pm, 2, raw, nullptr, st)) return rc;
        } else {
            const float* rows = pm.genomes;
            if (stage) {
                if (int rc = x256::launch_stage(b, pm, pm.count, staged, st)) return rc;
                rows = staged;
            }
            if (int rc = x256::launch_table(b, rows, pm.count, 2, raw, nullptr, st)) return rc;
        }
        tpop::Args args;
        args.sig = b->sig; args.px = b->px; args.bmax = b->bmax; args.smin = b->smin;
        args.T = T; args.tick = b->tick; args.phi = phi; args.fee = fee;
        args.raw = raw;
        args.adv = pa ? *pa : PopArgs{};
        args.tr = cols;
        const int64_t off = b0 * T;
        auto shift = [off](auto*& p) { if (p) p += off; };
        sgmm_trace& c = args.tr;
        shift(c.off_a); shift(c.off_b); shift(c.adv_a); shift(c.adv_b); shift(c.fill_buy); shift(c.fill_sell); shift(c.inventory);
        shift(c.cash); shift(c.reward); shift(c.pnl_reward); shift(c.inventory_reward); shift(c.fee_paid); shift(c.raw_a);
        shift(c.raw_b); shift(c.spread); shift(c.wealth); shift(c.cum_reward); shift(c.skew); shift(c.cum_fees);
        shift(c.unrealized_pnl);
        args.fitness = fitness + b0; args.trades = trades + b0;
        return pa ? tpop::launch_kernel<tpop::RawWalk20>(args, pm.count, st) : tpop::launch_kernel<tpop::RawWalk5>(args, pm.count, st);
    });
    if (rc) return rc;
    return release.done();
}

}  // namespace sgmm
