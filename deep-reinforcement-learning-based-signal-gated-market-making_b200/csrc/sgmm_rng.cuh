// sgmm_rng.cuh -- counter-based mutation noise (replaces the unseeded torch.randn_like of
// /root/reference/models/model.py:69).  Philox4x32-10 + Box-Muller whose log / sincos are built
// only from IEEE-exact operations (add, mul, fma, div, sqrt), so the device stream is bit-identical
// to the CPU oracle's and independent of the launch geometry:
//     noise(seed, generation, individual, element e) = normal4(key=seed, ctr=(e/4, ind_lo, ind_hi, gen))[e%4]
#pragma once
#include <stdint.h>
#include "sgmm_internal.h"

namespace sgmm {

__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

// ln(u), u = k*2^-24 in (0,1]
__device__ __forceinline__ float det_logf(float u)
{
    const uint32_t b = __float_as_uint(u);
    int e = (int)(b >> 23) - 127;
    float m = __uint_as_float((b & 0x007FFFFFu) | 0x3F800000u);
    if (m > 1.41421356f) { m = __fmul_rn(m, 0.5f); e += 1; }
    const float t = __fdiv_rn(__fadd_rn(m, -1.0f), __fadd_rn(m, 1.0f));
    const float t2 = __fmul_rn(t, t);
    float p = __fmaf_rn(t2, 0.11111111f, 0.14285715f);
    p = __fmaf_rn(t2, p, 0.2f);
    p = __fmaf_rn(t2, p, 0.33333334f);
    p = __fmul_rn(p, t2);
    float lm = __fmaf_rn(t, p, t);
    lm = __fadd_rn(lm, lm);
    return __fmaf_rn((float)e, 0.69314718f, lm);
}

// sin, cos of 2*pi*u, u = k*2^-24 in [0,1)
__device__ __forceinline__ void det_sincos2pi(float u, float& s, float& c)
{
    const float u4 = __fmul_rn(u, 4.0f);
    const int q = (int)u4;
    const float f = __fadd_rn(u4, -(float)q);
    const bool swap = f > 0.5f;
    const float g = swap ? __fadd_rn(1.0f, -f) : f;
    const float x = __fmul_rn(g, 1.57079633f);
    const float x2 = __fmul_rn(x, x);
    float sp = __fmaf_rn(x2, 2.7557319e-6f, -1.9841270e-4f);
    sp = __fmaf_rn(x2, sp, 8.3333333e-3f);
    sp = __fmaf_rn(x2, sp, -1.6666667e-1f);
    sp = __fmul_rn(sp, x2);
    const float sn = __fmaf_rn(x, sp, x);
    float cp = __fmaf_rn(x2, 2.4801587e-5f, -1.3888889e-3f);
    cp = __fmaf_rn(x2, cp, 4.1666668e-2f);
    cp = __fmaf_rn(x2, cp, -0.5f);
    const float cs = __fmaf_rn(x2, cp, 1.0f);
    const float s0 = swap ? cs : sn, c0 = swap ? sn : cs;
    switch (q) {
        case 0: s = s0;  c = c0;  break;
        case 1: s = c0;  c = -s0; break;
        case 2: s = -s0; c = -c0; break;
        default: s = -c0; c = s0; break;
    }
}

__device__ __forceinline__ void normal4(uint64_t seed, uint64_t generation, uint64_t individual,
                                        uint32_t block, float (&out)[4])
{
    uint32_t c[4] = { block, (uint32_t)individual, (uint32_t)(individual >> 32), (uint32_t)generation };
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const float u1 = __fmul_rn((float)((c[2 * h] >> 8) + 1u), 0x1p-24f);
        const float u2 = __fmul_rn((float)(c[2 * h + 1] >> 8), 0x1p-24f);
        const float r = __fsqrt_rn(__fmul_rn(-2.0f, det_logf(u1)));
        float s, co; det_sincos2pi(u2, s, co);
        out[2 * h] = __fmul_rn(r, co); out[2 * h + 1] = __fmul_rn(r, s);
    }
}

// where a genome value comes from: explicit [P,G] row, or master + sigma * noise
struct GenomeSource {
    const float* row;        // explicit genome row (or the master when seeded)
    bool seeded;
    float sigma;
    uint64_t seed, generation, individual;

    __device__ __forceinline__ float at(int64_t e) const
    {
        const float base = __ldg(row + e);
        if (!seeded) return base;
        float n[4]; normal4(seed, generation, individual, (uint32_t)(e >> 2), n);
        const float z = (e & 3) == 0 ? n[0] : (e & 3) == 1 ? n[1] : (e & 3) == 2 ? n[2] : n[3];
        return __fadd_rn(base, __fmul_rn(z, sigma));              // model.py:69-70: master + noise*sigma
    }
    // four consecutive elements starting at a multiple of 4
    __device__ __forceinline__ void at4(int64_t e0, float (&v)[4]) const
    {
        if (!seeded) {
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = __ldg(row + e0 + i);
            return;
        }
        float n[4]; normal4(seed, generation, individual, (uint32_t)(e0 >> 2), n);
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = __fadd_rn(__ldg(row + e0 + i), __fmul_rn(n[i], sigma));
    }
};

// device scalars of the GA (best child index, decayed sigma, generation) override the host values
__device__ __forceinline__ PopArgs resolve(const PopArgs& p)
{
    PopArgs r = p;
    if (p.first_index_dev) r.first_index += *p.first_index_dev;
    if (p.sigma_dev) r.sigma = *p.sigma_dev;
    if (p.generation_dev) r.generation = (uint64_t)(*p.generation_dev);
    return r;
}

__device__ __forceinline__ GenomeSource make_source(const PopArgs& p, int64_t i, int64_t G)
{
    GenomeSource g;
    g.seeded = (p.genomes == nullptr);
    g.row = g.seeded ? p.master : p.genomes + i * G;
    g.sigma = p.sigma; g.seed = p.seed; g.generation = p.generation;
    g.individual = (uint64_t)(p.first_index + i);
    return g;
}

// a GA sweep's children (SweepPop, sgmm_internal.h): individual i of the launch is child (first + i) % lambda of run
// (first + i) / lambda, drawn exactly as the solo GA of that run draws it
__device__ __forceinline__ SweepPop resolve(const SweepPop& p) { return p; }

__device__ __forceinline__ GenomeSource make_source(const SweepPop& p, int64_t i, int64_t G)
{
    const int64_t g = p.first + i, r = g / p.lambda;
    const GaDev* s = p.st + r;
    GenomeSource src;
    src.seeded = true;
    src.row = p.master + r * G;
    src.sigma = p.adv ? s->adv_sigma : s->sigma;
    src.seed = p.adv ? s->seed ^ ADV_SEED_FLIP : s->seed;
    src.generation = (uint64_t)s->generation;
    src.individual = (uint64_t)(g - r * p.lambda);
    return src;
}

// the source of individual i of a launch, device scalars resolved
template <class Pop>
__device__ __forceinline__ GenomeSource source_of(const Pop& p, int64_t i, int64_t G) { return make_source(resolve(p), i, G); }

}  // namespace sgmm
