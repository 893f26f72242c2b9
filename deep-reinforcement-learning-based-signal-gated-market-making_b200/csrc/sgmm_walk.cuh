// sgmm_walk.cuh -- the automata of the policy-table walks: maps {0..4} -> {0..4} (no adversary) and {0..19} -> {0..19}
// (with the adversary), their composition, the adversary's step of one bar and its displacement table.  Used by the
// walk kernels of sgmm_one.cu and by the population trace (sgmm_trace_pop.cu).
#pragma once
#include "sgmm_internal.h"
#include "sgmm_rng.cuh"
#include "sgmm_adversary.cuh"

namespace sgmm {
namespace one {

// maps {0..4} -> {0..4} packed 3 bits per entry
__device__ __forceinline__ uint32_t map_of(const uint8_t* n) { return n[0] | (n[1] << 3) | (n[2] << 6) | (n[3] << 9) | (n[4] << 12); }
__device__ __forceinline__ uint32_t map_at(uint32_t m, uint32_t e) { return (m >> (3u * e)) & 7u; }
// (g after f)[e] = g[f[e]]
__device__ __forceinline__ uint32_t map_then(uint32_t f, uint32_t g)
{
    return map_at(g, map_at(f, 0)) | (map_at(g, map_at(f, 1)) << 3) | (map_at(g, map_at(f, 2)) << 6) | (map_at(g, map_at(f, 3)) << 9) |
           (map_at(g, map_at(f, 4)) << 12);
}
constexpr uint32_t MAP_ID = 0u | (1u << 3) | (2u << 6) | (3u << 9) | (4u << 12);

// Maps {0..19} -> {0..19}: 20 entries of 5 bits, six per 32-bit word.
struct Map20 { uint32_t w[4]; };
__device__ __forceinline__ uint32_t m20_at(const Map20& m, uint32_t e)          // dynamic index
{
    const uint32_t hi = e >= 12u, w = hi ? (e >= 18u ? m.w[3] : m.w[2]) : (e >= 6u ? m.w[1] : m.w[0]);
    const uint32_t base = hi ? (e >= 18u ? 18u : 12u) : (e >= 6u ? 6u : 0u);
    return (w >> (5u * (e - base))) & 31u;
}
template <int S> __device__ __forceinline__ uint32_t m20_get(const Map20& m) { return (m.w[S / 6] >> (5 * (S % 6))) & 31u; }
template <int S> __device__ __forceinline__ void m20_set(Map20& m, uint32_t v) { m.w[S / 6] |= v << (5 * (S % 6)); }
template <int S = 0>
__device__ __forceinline__ void m20_then_rec(const Map20& f, const Map20& g, Map20& out)     // out[s] = g[f[s]]
{
    if constexpr (S < 20) { m20_set<S>(out, m20_at(g, m20_get<S>(f))); m20_then_rec<S + 1>(f, g, out); }
}
__device__ __forceinline__ Map20 m20_then(const Map20& f, const Map20& g) { Map20 o = {{0u, 0u, 0u, 0u}}; m20_then_rec(f, g, o); return o; }
template <int S = 0> __device__ __forceinline__ void m20_id_rec(Map20& m) { if constexpr (S < 20) { m20_set<S>(m, (uint32_t)S); m20_id_rec<S + 1>(m); } }
__device__ __forceinline__ Map20 m20_identity() { Map20 m = {{0u, 0u, 0u, 0u}}; m20_id_rec(m); return m; }
__device__ __forceinline__ Map20 m20_shfl_up(const Map20& m, int d)
{
    Map20 o;
#pragma unroll
    for (int i = 0; i < 4; ++i) o.w[i] = __shfl_up_sync(0xffffffffu, m.w[i], d);
    return o;
}

// the market maker's offset of one side, before the adversary's displacement (drl_engine.py:39, clamped to +-K_CLAMP)
__device__ __forceinline__ int mm_offset(float q) { return max(min(__float2int_rn(q), K_CLAMP), -K_CLAMP); }
// one bar's step from state st: displaced offsets, fills against the integer thresholds, next state
struct AdvStep { int oa, ob; bool fb, fs; uint32_t next; };
// (q: the q = raw*5 of the state's inventory at this bar)
__device__ __forceinline__ AdvStep adv_step_q(uint32_t st, float2 q, int2 k1, uint32_t at0, uint32_t at1, uint32_t at2)
{
    const uint32_t iv = st % 5u;
    const uint32_t e = table_lookup(at0, at1, at2, (int)st);
    AdvStep r;
    r.oa = mm_offset(q.x) + (int)(e & 3u) - 1;                                              // market_env.py:26-28
    r.ob = mm_offset(q.y) + (int)(e >> 2) - 1;
    r.fb = (iv < 4u) && (r.ob < k1.y);                                                     // :34,:37
    r.fs = (iv > 0u) && (r.oa < k1.x);                                                     // :35,:38
    r.next = (r.fs ? 10u : 0u) + (r.fb ? 5u : 0u) + iv + (r.fb ? 1u : 0u) - (r.fs ? 1u : 0u);
    return r;
}
__device__ __forceinline__ AdvStep adv_step(uint32_t st, const float2* __restrict__ code_t, int2 k1, uint32_t at0, uint32_t at1, uint32_t at2)
{
    return adv_step_q(st, code_t[st % 5u], k1, at0, at1, at2);
}
template <int S = 0>
__device__ __forceinline__ void bar_map_rec(Map20& m, const float2* __restrict__ code_t, int2 k1, uint32_t at0, uint32_t at1, uint32_t at2)
{
    if constexpr (S < 20) { m20_set<S>(m, adv_step((uint32_t)S, code_t, k1, at0, at1, at2).next); bar_map_rec<S + 1>(m, code_t, k1, at0, at1, at2); }
}

// the individual's adversary as its displacement table (sgmm_adversary.cuh), built in s_adv[3] (shared memory) by the
// first 20 threads; every thread of the block calls it
__device__ __forceinline__ void build_adv_table(const PopArgs& adv_in, int64_t ind, uint32_t* s_adv)
{
    const int tid = threadIdx.x;
    if (tid < 3) s_adv[tid] = 0u;
    __syncthreads();
    if (tid < 20) {
        const PopArgs advp = resolve(adv_in);
        const uint32_t e = adversary_entry(make_source(advp, ind, (int64_t)1250), tid);
        atomicOr(&s_adv[tid >> 3], e << ((tid & 7) * 4));
    }
    __syncthreads();
}

}  // namespace one
}  // namespace sgmm
