// sgmm_ga.cu -- device-side (1,lambda) evolution: NeuroEvolution.ask/tell and the generation loop
// of DRLEngine.train (/root/reference/models/model.py:59-76, Env/drl_engine.py:92-171) with no
// host round trip inside a generation.
//   ask       children are never materialised: the rollout kernel regenerates child i from
//             (master, sigma, seed, generation, i) with the counter-based noise of sgmm_rng.cuh
//   tell      argmax with numpy's semantics (first maximum, a NaN wins) -> master <- that child
//             (model.py:73-76); the adversary is told -fitness (drl_engine.py:123-125).  After sgmm_ga_set_parents:
//             the mu best children (device top-k) recombined into master + sigma * sum_k w_k eps_k instead; after
//             sgmm_ga_set_es: centered-rank utilities of every child, g = sum_i u_i eps_i / (lambda sigma), an Adam step
//   validate  rollout of the new master (== best child, drl_engine.py:129-140) with no adversary
//   select    keep-best-on-validation snapshot (:144-150), sigma halving after `patience` stale
//             generations (:155-160), history (:163-167)
// A sweep (sgmm_ga_create_sweep) advances K independent runs with the same launches: K*lambda children in one policy
// table and one walk (sgmm_one.cu), one tell block and one update block per run, the K new masters validated as one
// population.  Each run's state is its own GaDev (sgmm_internal.h) and history row; run r is bit-identical to the solo GA
// of its seed, phi, fee, sigma and patience.  A GA from sgmm_ga_create is the one-run case of the same kernels.
#include <cmath>
#include <new>
#include <vector>
#include "sgmm_internal.h"
#include "sgmm_rng.cuh"

namespace sgmm {

// The population's results live in ONE rank-blocked buffer so that a sharded generation needs a single all-gather:
//   block r (block_bytes each) = { double fitness[stride]; int32_t trades[stride]; pad }   individuals [r*stride, (r+1)*stride)
// With one rank there is one block and stride = pop_size.
struct Gather {
    char* base; int64_t stride; int64_t block_bytes;
    __host__ __device__ double* fit_block(int64_t r) const { return reinterpret_cast<double*>(base + r * block_bytes); }
    __host__ __device__ int32_t* trd_block(int64_t r) const { return reinterpret_cast<int32_t*>(base + r * block_bytes + stride * 8); }
    __device__ double fit(int64_t i) const { return fit_block(i / stride)[i % stride]; }
    __device__ int32_t trd(int64_t i) const { return trd_block(i / stride)[i % stride]; }
};

// numpy argmax over fitness (SIGN=+1) or over -fitness (SIGN=-1) of individuals first .. first+n-1: first maximum, first
// NaN wins.  Returns the index relative to `first`.
template <int SIGN>
__device__ int64_t block_argmax(const Gather& f, int64_t first, int64_t n, double* s_val, int64_t* s_idx)
{
    const int tid = threadIdx.x, nt = blockDim.x;
    double bv = 0.0; int64_t bi = -1; bool bnan = false;
    for (int64_t i = tid; i < n; i += nt) {
        const double v = SIGN > 0 ? f.fit(first + i) : -f.fit(first + i);
        const bool isn = (v != v);
        if (bi < 0) { bv = v; bi = i; bnan = isn; }
        else if (!bnan && (isn || v > bv)) { bv = v; bi = i; bnan = isn; }
    }
    s_val[tid] = bv; s_idx[tid] = bi;
    __syncthreads();
    for (int off = nt / 2; off >= 1; off >>= 1) {
        if (tid < off) {
            const double v2 = s_val[tid + off]; const int64_t i2 = s_idx[tid + off];
            const double v1 = s_val[tid]; const int64_t i1 = s_idx[tid];
            bool take = false;
            if (i2 >= 0) {
                if (i1 < 0) take = true;
                else {
                    const bool n1 = (v1 != v1), n2 = (v2 != v2);
                    if (n1 && n2) take = i2 < i1;
                    else if (n2) take = true;
                    else if (n1) take = false;
                    else take = (v2 > v1) || (v2 == v1 && i2 < i1);
                }
            }
            if (take) { s_val[tid] = v2; s_idx[tid] = i2; }
        }
        __syncthreads();
    }
    const int64_t r = s_idx[0];
    __syncthreads();
    return r;
}

// One block per run: block r tells run r the results of its children [r*pop, (r+1)*pop) and moves run r's masters (rows r
// of mm_masters [runs][G] and adv_masters [runs][1250]) to the best child.
__global__ void __launch_bounds__(256) ga_tell_kernel(GaDev* runs, const Gather fit, int64_t pop,
                                                      float* mm_masters, int64_t G, float* adv_masters, int use_arl)
{
    __shared__ double s_val[256];
    __shared__ int64_t s_idx[256];
    const int64_t run = blockIdx.x, first = run * pop;
    GaDev* st = runs + run;
    float* mm_master = mm_masters + run * G;
    float* adv_master = adv_masters + run * 1250;
    const int64_t best = block_argmax<+1>(fit, first, pop, s_val, s_idx);
    int64_t abest = 0;
    if (use_arl) abest = block_argmax<-1>(fit, first, pop, s_val, s_idx);
    const uint64_t gen = (uint64_t)st->generation, seed = st->seed;
    const float sigma = st->sigma, asigma = st->adv_sigma;
    // master <- child[best]  (regenerated: master + sigma*noise, element-wise, in place)
    for (int64_t e = threadIdx.x; e < G; e += blockDim.x) {
        float n[4]; normal4(seed, gen, (uint64_t)best, (uint32_t)(e >> 2), n);
        mm_master[e] = __fadd_rn(mm_master[e], __fmul_rn(n[e & 3], sigma));
    }
    if (use_arl) {
        for (int64_t e = threadIdx.x; e < 1250; e += blockDim.x) {
            float n[4]; normal4(seed ^ ADV_SEED_FLIP, gen, (uint64_t)abest, (uint32_t)(e >> 2), n);
            adv_master[e] = __fadd_rn(adv_master[e], __fmul_rn(n[e & 3], asigma));
        }
    }
    if (threadIdx.x == 0) {
        st->best_idx = best; st->adv_best_idx = abest;
        st->train_f = fit.fit(first + best); st->train_trades = fit.trd(first + best);
    }
}

// One block per run: run r's validation result val_f[r] / val_t[r], masters row r, history row r ([runs][max_gen]).
__global__ void __launch_bounds__(256) ga_update_kernel(GaDev* runs, const double* val_fs, const int32_t* val_ts,
                                                        const float* mm_masters, float* best_masters, int64_t G,
                                                        int use_arl, int max_gen,
                                                        double* h_train_f, double* h_val_f, int32_t* h_train_t,
                                                        int32_t* h_val_t, float* h_sigma)
{
    __shared__ int improved;
    const int64_t run = blockIdx.x, row = run * max_gen;
    GaDev* st = runs + run;
    const double* val_f = val_fs + run;
    const int32_t* val_t = val_ts + run;
    const float* mm_master = mm_masters + run * G;
    float* best_master = best_masters + run * G;
    if (threadIdx.x == 0) {
        const double v = *val_f;
        improved = (v > st->best_val) ? 1 : 0;                     // drl_engine.py:144 (NaN never improves)
    }
    __syncthreads();
    if (improved) for (int64_t e = threadIdx.x; e < G; e += blockDim.x) best_master[e] = mm_master[e];   // :149
    __syncthreads();
    if (threadIdx.x == 0) {
        const int g = st->generation;
        if (g < max_gen) {                                          // :163-167 (sigma logged before decay)
            h_train_f[row + g] = st->train_f; h_val_f[row + g] = *val_f; h_train_t[row + g] = st->train_trades;
            h_val_t[row + g] = *val_t; h_sigma[row + g] = st->sigma;
        }
        if (improved) { st->best_val = *val_f; st->stale = 0; } else st->stale += 1;     // :145-152
        if (st->stale >= st->patience) {                            // :155-160
            st->sigma = __fmul_rn(st->sigma, 0.5f);
            if (use_arl) st->adv_sigma = __fmul_rn(st->adv_sigma, 0.5f);
            st->stale = 0;
        }
        st->generation = g + 1;
    }
}

// ---- truncation selection (sgmm_ga_set_parents): the mu best children of a run, in rank order, recombined into the new
// master m + sigma * sum_k w_k eps_k.  The rank order is ga_tell_kernel's: NaN first, then descending fitness (adversary:
// descending -fitness), ties to the lower index, -0.0 == +0.0; with mu = 1 parent 0 is block_argmax's child.
constexpr int SELECT_THREADS = 512;
constexpr int RECOMBINE_THREADS = 64;

// Order-preserving 64-bit key of a fitness value, larger = ranked first: NaN is the maximum, -0.0 is canonicalised and
// SIGN = -1 ranks -fitness.  Every real key lies in [0x000F..F, 0xFFF0..0], so 0 is free for padding.
template <int SIGN>
__device__ __forceinline__ uint64_t rank_key(double v)
{
    if (v != v) return ~0ull;
    uint64_t b = (uint64_t)__double_as_longlong(v == 0.0 ? 0.0 : v);
    b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
    return SIGN > 0 ? b : ~b;
}

// Visits the children first .. first+n-1 of the gather buffer in index order, nt at a time, without a division per child:
// every thread of the block makes every call (the loop bounds are uniform), thread t with child base + t, or with
// valid == false past the end.  f(i, key, valid) gets the index relative to `first`.
template <int SIGN, class F>
__device__ __forceinline__ void for_children(const Gather& g, int64_t first, int64_t n, F&& f)
{
    const int64_t end = first + n;
    for (int64_t b = first / g.stride; b * g.stride < end; ++b) {
        const int64_t b0 = b * g.stride, lo = max(first, b0), hi = min(end, b0 + g.stride);
        const double* fb = g.fit_block(b);
        for (int64_t base = lo; base < hi; base += blockDim.x) {
            const int64_t gi = base + threadIdx.x;
            const bool valid = gi < hi;
            f(gi - first, valid ? rank_key<SIGN>(fb[gi - b0]) : 0ull, valid);
        }
    }
}

struct SelectSmem {
    uint64_t key[SGMM_MAX_PARENTS];
    int64_t idx[SGMM_MAX_PARENTS];
    int hist[256];
    int warp_ties[SELECT_THREADS / 32];
    int digit, k, count, ties_seen;
};

// The first mu children of the rank order of children first .. first+n-1, written to out[0..mu) (indices relative to
// `first`); returns out[0].  A radix select (8 passes of 8-bit digit histograms) finds the mu-th key; every key above it
// and the first keys equal to it in index order are kept, then sorted by (key descending, index ascending).
template <int SIGN>
__device__ int64_t select_parents(const Gather& f, int64_t first, int64_t n, int mu, SelectSmem& s, int64_t* out)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint64_t prefix = 0, mask = 0;
    int k = mu;                                                     // rank of the wanted key among those matching prefix
    for (int shift = 56; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += blockDim.x) s.hist[i] = 0;
        __syncthreads();
        for_children<SIGN>(f, first, n, [&](int64_t, uint64_t key, bool valid) {
            if (valid && (key & mask) == prefix) atomicAdd(&s.hist[(key >> shift) & 0xFF], 1);
        });
        __syncthreads();
        if (warp == 0) {                                            // lane l holds digits 255-8l .. 248-8l, top down
            int c[8], sum = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = s.hist[255 - 8 * lane - j]; sum += c[j]; }
            int incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= o) incl += y;
            }
            int cum = incl - sum;
            if (cum < k && k <= incl) {
                bool found = false;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (!found && cum + c[j] >= k) { s.digit = 255 - 8 * lane - j; s.k = k - cum; found = true; }
                    if (!found) cum += c[j];
                }
            }
        }
        __syncthreads();
        prefix |= (uint64_t)s.digit << shift; mask |= 0xFFull << shift; k = s.k;
    }
    // prefix is the mu-th key; k of the keys equal to it are parents, the first k in index order
    if (tid == 0) { s.count = 0; s.ties_seen = 0; }
    __syncthreads();
    for_children<SIGN>(f, first, n, [&](int64_t i, uint64_t key, bool valid) {
        const bool tie = valid && key == prefix;
        const unsigned ties = __ballot_sync(0xFFFFFFFFu, tie);
        if (lane == 0) s.warp_ties[warp] = __popc(ties);
        __syncthreads();
        int before = s.ties_seen + __popc(ties & ((1u << lane) - 1u));
        for (int w = 0; w < warp; ++w) before += s.warp_ties[w];
        if ((valid && key > prefix) || (tie && before < k)) {
            const int slot = atomicAdd(&s.count, 1);
            s.key[slot] = key; s.idx[slot] = i;
        }
        __syncthreads();
        if (tid == 0) for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s.ties_seen += s.warp_ties[w];
        __syncthreads();
    });
    int S = 1;
    while (S < mu) S <<= 1;
    for (int i = mu + tid; i < S; i += blockDim.x) { s.key[i] = 0; s.idx[i] = INT64_MAX; }   // padding sorts last
    __syncthreads();
    for (int size = 2; size <= S; size <<= 1) {                     // bitonic sort: (key descending, index ascending)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = tid; t < S / 2; t += blockDim.x) {
                const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
                const uint64_t kl = s.key[lo], kh = s.key[hi];
                const int64_t il = s.idx[lo], ih = s.idx[hi];
                const bool hi_first = kh > kl || (kh == kl && ih < il);
                if (hi_first == ((lo & size) == 0)) { s.key[lo] = kh; s.key[hi] = kl; s.idx[lo] = ih; s.idx[hi] = il; }
            }
            __syncthreads();
        }
    }
    for (int i = tid; i < mu; i += blockDim.x) out[i] = s.idx[i];
    const int64_t best = s.idx[0];
    __syncthreads();
    return best;
}

// One block per run: run r's parents (rows r of mm_parents / adv_parents [runs][mu]) and its best child's state, as
// ga_tell_kernel records it.  The masters are left to ga_recombine_kernel.
__global__ void __launch_bounds__(SELECT_THREADS) ga_select_kernel(GaDev* runs, const Gather fit, int64_t pop, int mu,
                                                                   int64_t* mm_parents, int64_t* adv_parents, int use_arl)
{
    __shared__ SelectSmem s;
    const int64_t run = blockIdx.x, first = run * pop;
    GaDev* st = runs + run;
    const int64_t best = select_parents<+1>(fit, first, pop, mu, s, mm_parents + run * mu);
    int64_t abest = 0;
    if (use_arl) abest = select_parents<-1>(fit, first, pop, mu, s, adv_parents + run * mu);
    if (threadIdx.x == 0) {
        st->best_idx = best; st->adv_best_idx = abest;
        st->train_f = fit.fit(first + best); st->train_trades = fit.trd(first + best);
    }
}

// Grid (runs, quad blocks): thread q of run r owns elements 4q .. 4q+3 of one master (quad blocks [0, mm_blocks) the
// market maker's [runs][G], the rest the adversary's [runs][1250]) and regenerates the same normal4 block of every parent:
//   acc = w0*eps_0;  acc = fma(w_k, eps_k, acc) for k = 1 .. mu-1 in rank order;  m += acc*sigma
// With w = [1] this is ga_tell_kernel's master + noise*sigma bit for bit.  Each thread updates only its own elements.
__global__ void __launch_bounds__(RECOMBINE_THREADS) ga_recombine_kernel(const GaDev* runs, int mu, const float* w,
                                                                         const int64_t* mm_parents, const int64_t* adv_parents,
                                                                         float* mm_masters, int64_t G, float* adv_masters,
                                                                         int mm_blocks)
{
    const int64_t run = blockIdx.x;
    const GaDev* st = runs + run;
    const bool adv = (int)blockIdx.y >= mm_blocks;
    const int64_t n = adv ? 1250 : G;
    const int64_t q = (int64_t)(adv ? blockIdx.y - mm_blocks : blockIdx.y) * blockDim.x + threadIdx.x;
    if (4 * q >= n) return;
    const int64_t* par = (adv ? adv_parents : mm_parents) + run * mu;
    float* m = adv ? adv_masters + run * 1250 : mm_masters + run * G;
    const uint64_t seed = adv ? st->seed ^ ADV_SEED_FLIP : st->seed, gen = (uint64_t)st->generation;
    const float sigma = adv ? st->adv_sigma : st->sigma;
    float acc[4];
    {
        float e[4]; normal4(seed, gen, (uint64_t)par[0], (uint32_t)q, e);
        const float w0 = w[0];
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i] = __fmul_rn(w0, e[i]);
    }
    for (int k = 1; k < mu; ++k) {
        float e[4]; normal4(seed, gen, (uint64_t)par[k], (uint32_t)q, e);
        const float wk = w[k];
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[i] = __fmaf_rn(wk, e[i], acc[i]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (4 * q + i < n) m[4 * q + i] = __fadd_rn(m[4 * q + i], __fmul_rn(acc[i], sigma));
}

// ---- natural-gradient evolution strategy (sgmm_ga_set_es): centered-rank utilities of all lambda children, the noise-
// weighted sum g = sum_i u_i eps_i / (lambda sigma) in a fixed order, and an Adam ascent step on the master.
//   rank      r_i = child i's position in ga_select_kernel's order (NaN first, then descending fitness -- the adversary's
//             ascending --, ties to the lower index, -0.0 == +0.0);  u_i = fl(fl((float)(lambda-1-r_i) / (float)(lambda-1)) - 0.5f)
//   sum       index order, segments of ES_SEGMENT children: acc = u_i*eps_i for a segment's first child, then fmaf(u_i, eps_i,
//             acc); the segment sums are combined by a pairwise tree ((s0+s1), (s2+s3), ...; an odd last one moves up)
//   gradient  g = fl(S * fl(1 / fl((float)lambda * sigma))), sigma the run's device sigma of this generation
//   Adam      p1 *= b1, p2 *= b2 (running products from 1, once per generation);  m = b1*m + (1-b1)*g;  v = b2*v + (1-b2)*g*g;
//             theta += lr * ((m / (1-p1)) / (sqrt(v / (1-p2)) + eps)), every operation one binary32 rounding
// The segment length is part of the definition, not of the launch.
constexpr int ES_SEGMENT = 256;
constexpr int ES_RANK_THREADS = 256;
constexpr int ES_GRAD_THREADS = 256;
constexpr int ES_GRAD_QUADS = 16;                                   // quads (64 elements) per gradient block
constexpr int ES_GRAD_CHUNK = 64;                                   // children per noise chunk of a gradient block
constexpr int ES_ADAM_THREADS = 256;
constexpr float ES_B1 = 0.9f, ES_B2 = 0.999f, ES_EPS = 1e-8f;

// Block (run, t) ranks run r's children t*256 .. t*256+255 in one direction by counting the children ranked before each
// (every key above it, and the equal keys of lower index), reading all the run's keys tile by tile through for_children.
template <int SIGN>
__device__ int64_t es_rank(const Gather& f, int64_t first, int64_t n, int64_t i, uint64_t* s_key, int64_t* s_j0)
{
    const uint64_t ki = i < n ? rank_key<SIGN>(f.fit(first + i)) : 0ull;
    int64_t before = 0;
    for_children<SIGN>(f, first, n, [&](int64_t j, uint64_t key, bool valid) {
        s_key[threadIdx.x] = key;                                   // the tile: children j0 .. j0+cnt-1 (a valid prefix)
        if (threadIdx.x == 0) *s_j0 = j;
        const int cnt = __syncthreads_count(valid);
        const int64_t j0 = *s_j0;
        const int lim = (int)max((int64_t)0, min((int64_t)cnt, i - j0));   // tile entries of lower index than i
        int c = 0;
        for (int k = 0; k < lim; ++k) c += s_key[k] >= ki ? 1 : 0;
        for (int k = lim; k < cnt; ++k) c += s_key[k] > ki ? 1 : 0;
        before += c;
        __syncthreads();
    });
    return before;
}

__device__ __forceinline__ float es_utility(int64_t r, int64_t n)
{
    return __fsub_rn(__fdiv_rn((float)(n - 1 - r), (float)(n - 1)), 0.5f);
}

// Grid (runs, ceil(lambda/256)): utilities u[runs][lambda] (and adv_u under use_arl), the best child's state as
// ga_select_kernel records it, and the run's Adam powers (block 0).
__global__ void __launch_bounds__(ES_RANK_THREADS) es_rank_kernel(GaDev* runs, const Gather fit, int64_t pop, float* u,
                                                                   float* adv_u, float* pows, int use_arl)
{
    __shared__ uint64_t s_key[ES_RANK_THREADS];
    __shared__ int64_t s_j0;
    const int64_t run = blockIdx.x, first = run * pop;
    const int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
    GaDev* st = runs + run;
    const int64_t r = es_rank<+1>(fit, first, pop, i, s_key, &s_j0);
    if (i < pop) {
        u[run * pop + i] = es_utility(r, pop);
        if (r == 0) {
            st->best_idx = i;
            st->train_f = fit.fit(first + i); st->train_trades = fit.trd(first + i);
            if (!use_arl) st->adv_best_idx = 0;
        }
    }
    if (use_arl) {
        const int64_t ra = es_rank<-1>(fit, first, pop, i, s_key, &s_j0);
        if (i < pop) {
            adv_u[run * pop + i] = es_utility(ra, pop);
            if (ra == 0) st->adv_best_idx = i;
        }
    }
    if (blockIdx.y == 0 && threadIdx.x == 0) {
        pows[2 * run] = __fmul_rn(pows[2 * run], ES_B1);
        pows[2 * run + 1] = __fmul_rn(pows[2 * run + 1], ES_B2);
    }
}

// Grid (runs, quad blocks, segments): block (r, b, s) owns ES_GRAD_QUADS element quads of one master (quad blocks
// [0, mm_blocks) the market maker's G elements, the rest the adversary's 1250) and segment s of run r's children.  Its
// threads regenerate the noise of ES_GRAD_CHUNK children at a time into shared memory; thread e < 64 then chains element
// e's fmaf over those children in index order.  The segment sum goes to part[r][s][element].
__global__ void __launch_bounds__(ES_GRAD_THREADS) es_grad_kernel(const GaDev* runs, int64_t pop, const float* u,
                                                                   const float* adv_u, float* part, float* adv_part,
                                                                   int64_t G, int mm_blocks)
{
    __shared__ float4 s_eps[ES_GRAD_CHUNK][ES_GRAD_QUADS];
    __shared__ float s_u[ES_GRAD_CHUNK];
    const int64_t run = blockIdx.x, seg = blockIdx.z, nseg = gridDim.z;
    const GaDev* st = runs + run;
    const bool adv = (int)blockIdx.y >= mm_blocks;
    const int64_t n = adv ? 1250 : G;
    const int64_t q0 = (int64_t)(adv ? blockIdx.y - mm_blocks : blockIdx.y) * ES_GRAD_QUADS;
    const float* ur = (adv ? adv_u : u) + run * pop;
    const uint64_t seed = adv ? st->seed ^ ADV_SEED_FLIP : st->seed, gen = (uint64_t)st->generation;
    const int64_t c0 = seg * ES_SEGMENT, c1 = min(pop, c0 + ES_SEGMENT);
    const int e = threadIdx.x;
    const int64_t elem = 4 * q0 + e;
    float acc = 0.0f;
    for (int64_t cb = c0; cb < c1; cb += ES_GRAD_CHUNK) {
        const int nc = (int)min((int64_t)ES_GRAD_CHUNK, c1 - cb);
        for (int t = threadIdx.x; t < ES_GRAD_CHUNK * ES_GRAD_QUADS; t += blockDim.x) {
            const int c = t / ES_GRAD_QUADS, qi = t % ES_GRAD_QUADS;
            const int64_t q = q0 + qi;
            if (c < nc && 4 * q < n) {
                float z[4]; normal4(seed, gen, (uint64_t)(cb + c), (uint32_t)q, z);
                s_eps[c][qi] = make_float4(z[0], z[1], z[2], z[3]);
            }
        }
        if (threadIdx.x < nc) s_u[threadIdx.x] = ur[cb + threadIdx.x];
        __syncthreads();
        if (e < 4 * ES_GRAD_QUADS) {
            const float* col = reinterpret_cast<const float*>(&s_eps[0][0]) + e;
            for (int c = 0; c < nc; ++c) {
                const float x = col[c * 4 * ES_GRAD_QUADS], w = s_u[c];
                acc = (cb + c == c0) ? __fmul_rn(w, x) : __fmaf_rn(w, x, acc);
            }
        }
        __syncthreads();
    }
    if (e < 4 * ES_GRAD_QUADS && elem < n) (adv ? adv_part + run * nseg * 1250 : part + run * nseg * G)[seg * n + elem] = acc;
}

// Grid (runs, element blocks): thread (r, e) combines element e's segment sums of run r by the pairwise tree (in place in
// part[r][.][e]), scales them into the gradient and takes the Adam step on the master (blocks [0, mm_blocks) the market
// maker's G elements, the rest the adversary's 1250, from its own utilities and adv_sigma).
__global__ void __launch_bounds__(ES_ADAM_THREADS) es_adam_kernel(const GaDev* runs, int64_t pop, int nseg, float lr,
                                                                   const float* pows, float* part, float* adv_part,
                                                                   float* grad, float* adv_grad, float* mom, float* adv_mom,
                                                                   float* vel, float* adv_vel, float* mm_masters,
                                                                   float* adv_masters, int64_t G, int mm_blocks)
{
    const int64_t run = blockIdx.x;
    const GaDev* st = runs + run;
    const bool adv = (int)blockIdx.y >= mm_blocks;
    const int64_t n = adv ? 1250 : G;
    const int64_t e = (int64_t)(adv ? blockIdx.y - mm_blocks : blockIdx.y) * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float* p = (adv ? adv_part + run * (int64_t)nseg * 1250 : part + run * (int64_t)nseg * G) + e;
    for (int len = nseg; len > 1; len = (len + 1) >> 1) {
        for (int k = 0; 2 * k + 1 < len; ++k) p[k * n] = __fadd_rn(p[2 * k * n], p[(2 * k + 1) * n]);
        if (len & 1) p[(len >> 1) * n] = p[(len - 1) * n];
    }
    const float sigma = adv ? st->adv_sigma : st->sigma;
    const float g = __fmul_rn(p[0], __fdiv_rn(1.0f, __fmul_rn((float)pop, sigma)));
    const int64_t o = run * n + e;
    float* m = (adv ? adv_mom : mom) + o;
    float* v = (adv ? adv_vel : vel) + o;
    float* th = (adv ? adv_masters : mm_masters) + o;
    (adv ? adv_grad : grad)[o] = g;
    const float p1 = pows[2 * run], p2 = pows[2 * run + 1];
    const float mn = __fadd_rn(__fmul_rn(ES_B1, *m), __fmul_rn(__fsub_rn(1.0f, ES_B1), g));
    const float vn = __fadd_rn(__fmul_rn(ES_B2, *v), __fmul_rn(__fsub_rn(1.0f, ES_B2), __fmul_rn(g, g)));
    const float mh = __fdiv_rn(mn, __fsub_rn(1.0f, p1));
    const float vh = __fdiv_rn(vn, __fsub_rn(1.0f, p2));
    *m = mn; *v = vn;
    *th = __fadd_rn(*th, __fmul_rn(lr, __fdiv_rn(mh, __fadd_rn(__fsqrt_rn(vh), ES_EPS))));
}

}  // namespace sgmm

using namespace sgmm;

struct sgmm_ga {
    int device = 0;
    sgmm_ga_config cfg{};
    int32_t runs = 1;                 // independent runs advanced together: [runs] rows of every per-run buffer
    bool sweep = false;               // from sgmm_ga_create_sweep: children on the sweep's policy-table path (sgmm_one.cu)
    int64_t G = 0, capacity = 0;
    float* mm_master = nullptr; float* adv_master = nullptr; float* best_master = nullptr;   // [runs][G], [runs][1250], [runs][G]
    sgmm::Gather gather{nullptr, 0, 0}; int64_t n_blocks = 1, my_block = 0;
    double* my_fit() const { return gather.fit_block(my_block); }          // this rank's slice: children [shard_first, +shard_count)
    int32_t* my_trd() const { return gather.trd_block(my_block); }
    double* val_fit = nullptr; int32_t* val_trd = nullptr;                  // [runs]
    GaDev* st = nullptr;                                                    // [runs]
    double* h_train_f = nullptr; double* h_val_f = nullptr; int32_t* h_train_t = nullptr; int32_t* h_val_t = nullptr;
    float* h_sigma = nullptr;                                               // [runs][max_generations]
    // truncation selection (sgmm_ga_set_parents): weights != nullptr selects ga_select_kernel + ga_recombine_kernel
    int32_t parents = 1;
    float* weights = nullptr;                                               // [parents]
    int64_t* mm_parents = nullptr; int64_t* adv_parents = nullptr;          // [runs][parents]
    // evolution strategy (sgmm_ga_set_es): es_lr > 0 selects es_rank_kernel + es_grad_kernel + es_adam_kernel
    float es_lr = 0.0f;
    int32_t es_nseg = 0;                                                    // ceil(lambda / ES_SEGMENT)
    float* es_u = nullptr; float* es_adv_u = nullptr;                       // [runs][lambda]
    float* es_part = nullptr; float* es_adv_part = nullptr;                 // [runs][nseg][G], [runs][nseg][1250]
    float* es_grad = nullptr; float* es_adv_grad = nullptr;                 // [runs][G], [runs][1250]
    float* es_m = nullptr; float* es_adv_m = nullptr;                       // Adam moments, as the gradients
    float* es_v = nullptr; float* es_adv_v = nullptr;
    float* es_pow = nullptr;                                                // [runs][2]: b1^t, b2^t
    // training objective (sgmm_ga_set_objective): what the population and validation rollouts write as fitness
    int32_t objective = SGMM_OBJECTIVE_REWARD;
    bool started = false;                                                   // a generation phase has been enqueued
};

namespace {
// device buffers of ga->runs runs, initial states `init` [runs] and HOST masters [runs][G] / [runs][1250] (adv may be NULL)
int ga_allocate(sgmm_ga* ga, const GaDev* init, const float* mm_masters, const float* adv_masters, cudaStream_t st)
{
    DeviceGuard guard(ga->device);
    const size_t R = (size_t)ga->runs, G = (size_t)ga->G, cap = (size_t)ga->capacity, mg = (size_t)ga->cfg.max_generations;
    int rc = SGMM_OK;
    if (!rc) rc = check_cuda(cudaMalloc(&ga->mm_master, R * G * sizeof(float)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->best_master, R * G * sizeof(float)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->adv_master, R * 1250 * sizeof(float)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->gather.base, cap), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->val_fit, R * sizeof(double)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->val_trd, R * sizeof(int32_t)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->st, R * sizeof(GaDev)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_train_f, R * mg * sizeof(double)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_val_f, R * mg * sizeof(double)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_train_t, R * mg * sizeof(int32_t)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_val_t, R * mg * sizeof(int32_t)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_sigma, R * mg * sizeof(float)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMemcpyAsync(ga->st, init, R * sizeof(GaDev), cudaMemcpyHostToDevice, st), "H2D ga state");
    if (!rc) rc = check_cuda(cudaMemcpyAsync(ga->mm_master, mm_masters, R * G * sizeof(float), cudaMemcpyHostToDevice, st), "H2D master");
    if (!rc) rc = check_cuda(cudaMemcpyAsync(ga->best_master, mm_masters, R * G * sizeof(float), cudaMemcpyHostToDevice, st), "H2D master");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->adv_master, 0, R * 1250 * sizeof(float), st), "memset");
    if (!rc && adv_masters) rc = check_cuda(cudaMemcpyAsync(ga->adv_master, adv_masters, R * 1250 * sizeof(float), cudaMemcpyHostToDevice, st), "H2D adv master");
    // history of generations not yet run reads as zeros (the history read-backs additionally clamp n to the generations completed)
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_train_f, 0, R * mg * sizeof(double), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_val_f, 0, R * mg * sizeof(double), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_train_t, 0, R * mg * sizeof(int32_t), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_val_t, 0, R * mg * sizeof(int32_t), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_sigma, 0, R * mg * sizeof(float), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->gather.base, 0, cap, st), "memset");
    if (!rc) rc = check_cuda(cudaStreamSynchronize(st), "ga_create");
    return rc;
}

GaDev initial_state(float sigma, int32_t patience, uint64_t seed, double phi, double fee)
{
    GaDev s{};
    s.generation = 0; s.stale = 0; s.sigma = sigma; s.adv_sigma = sigma;
    s.best_val = -INFINITY;                                         // drl_engine.py:84
    s.patience = patience; s.seed = seed; s.phi = phi; s.fee = fee;
    return s;
}

// the run-less entries address run 0 and are refused on a handle of several runs
int single_run(const sgmm_ga* ga, const char* what)
{
    if (ga->runs == 1) return SGMM_OK;
    set_error("%s: this GA is a sweep of %d runs; use the per-run entry sgmm_ga_run_%s", what, (int)ga->runs,
              what + sizeof("sgmm_ga_") - 1);
    return SGMM_ERR_INVALID;
}

void es_free(sgmm_ga* ga)
{
    float** bufs[] = {&ga->es_u, &ga->es_adv_u, &ga->es_part, &ga->es_adv_part, &ga->es_grad, &ga->es_adv_grad,
                      &ga->es_m, &ga->es_adv_m, &ga->es_v, &ga->es_adv_v, &ga->es_pow};
    for (float** b : bufs) { cudaFree(*b); *b = nullptr; }
    ga->es_lr = 0.0f; ga->es_nseg = 0;
}

int check_run(const sgmm_ga* ga, int32_t run)
{
    if (run >= 0 && run < ga->runs) return SGMM_OK;
    set_error("run %d out of range: this GA has %d run(s)", (int)run, (int)ga->runs);
    return SGMM_ERR_INVALID;
}
}  // namespace

extern "C" {

int sgmm_ga_create(sgmm_ga** out, const sgmm_ga_config* cfg, const float* mm_master, const float* adv_master,
                   int device, void* stream)
{
    if (!out || !cfg || !mm_master) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    *out = nullptr;
    if (cfg->hidden != 32 && cfg->hidden != 256) { set_error("hidden=%d: GA rollouts are built for H=32 and H=256", cfg->hidden); return SGMM_ERR_UNSUPPORTED; }
    if (cfg->hidden == 256 && cfg->precision == SGMM_PRECISION_F32) { set_error("hidden=256: pass precision=SGMM_PRECISION_EXACT (bit-exact SGMM-F32 order) or SGMM_PRECISION_BF16 (tensor cores)"); return SGMM_ERR_UNSUPPORTED; }
    if (cfg->precision != SGMM_PRECISION_F32 && cfg->precision != SGMM_PRECISION_BF16 && cfg->precision != SGMM_PRECISION_TF32 && cfg->precision != SGMM_PRECISION_F16 && cfg->precision != SGMM_PRECISION_EXACT) { set_error("unknown precision %d", cfg->precision); return SGMM_ERR_INVALID; }
    if (cfg->hidden == 256 && cfg->use_arl && cfg->precision != SGMM_PRECISION_EXACT && cfg->precision != SGMM_PRECISION_BF16) { set_error("use_arl at hidden=256: pass precision=SGMM_PRECISION_BF16 (tensor cores) or SGMM_PRECISION_EXACT"); return SGMM_ERR_UNSUPPORTED; }
    if (cfg->pop_size <= 0 || cfg->shard_first < 0 || cfg->shard_count < 0 ||
        cfg->shard_first + cfg->shard_count > cfg->pop_size) { set_error("bad population / shard bounds"); return SGMM_ERR_INVALID; }
    const int64_t stride = cfg->shard_stride > 0 ? cfg->shard_stride : cfg->pop_size;
    if (cfg->shard_stride < 0 || (cfg->shard_count > 0 && cfg->shard_first % stride != 0) || cfg->shard_count > stride ||
        (cfg->shard_stride == 0 && cfg->shard_count != cfg->pop_size)) {
        set_error("bad shard_stride: shards are blocks of shard_stride individuals, shard_first a multiple of it, shard_count <= it "
                  "(0 = unsharded)"); return SGMM_ERR_INVALID;
    }
    if (cfg->use_arl && !adv_master) { set_error("use_arl needs an adversary master"); return SGMM_ERR_INVALID; }
    if (cfg->max_generations <= 0) { set_error("max_generations must be > 0"); return SGMM_ERR_INVALID; }
    sgmm_ga* ga = new (std::nothrow) sgmm_ga();
    if (!ga) { set_error("out of host memory"); return SGMM_ERR_NOMEM; }
    ga->device = device; ga->cfg = *cfg; ga->G = genome_len(cfg->hidden);
    ga->n_blocks = (cfg->pop_size + stride - 1) / stride; ga->my_block = cfg->shard_first / stride;
    if (ga->my_block >= ga->n_blocks) ga->my_block = ga->n_blocks - 1;     // an empty trailing shard (shard_count == 0)
    ga->gather.stride = stride; ga->gather.block_bytes = (stride * 12 + 15) / 16 * 16;
    ga->capacity = ga->n_blocks * ga->gather.block_bytes;
    const GaDev init = initial_state(cfg->sigma, cfg->patience, cfg->seed, cfg->phi, cfg->fee_rate);
    if (int rc = ga_allocate(ga, &init, mm_master, adv_master, (cudaStream_t)stream)) { sgmm_ga_destroy(ga); return rc; }
    *out = ga;
    return SGMM_OK;
}

int sgmm_ga_create_sweep(sgmm_ga** out, const sgmm_ga_config* cfg, int32_t runs, const sgmm_ga_run* run,
                         const float* mm_masters, const float* adv_masters, int device, void* stream)
{
    if (!out) { set_error("out is NULL"); return SGMM_ERR_INVALID; }
    *out = nullptr;
    if (!cfg) { set_error("cfg is NULL"); return SGMM_ERR_INVALID; }
    if (cfg->hidden != 32) { set_error("hidden=%d: a GA sweep runs hidden=32 only (hidden=256 GAs run one at a time: sgmm_ga_create)", cfg->hidden); return SGMM_ERR_UNSUPPORTED; }
    if (cfg->precision != SGMM_PRECISION_F32 && cfg->precision != SGMM_PRECISION_EXACT) {
        if (cfg->precision == SGMM_PRECISION_BF16 || cfg->precision == SGMM_PRECISION_TF32 || cfg->precision == SGMM_PRECISION_F16) {
            set_error("precision %d: a GA sweep runs the exact path only (SGMM_PRECISION_F32 / SGMM_PRECISION_EXACT); tensor-core GAs run one at a time: sgmm_ga_create", cfg->precision);
            return SGMM_ERR_UNSUPPORTED;
        }
        set_error("unknown precision %d", cfg->precision); return SGMM_ERR_INVALID;
    }
    if (runs <= 0) { set_error("runs=%d: a sweep needs at least one run", (int)runs); return SGMM_ERR_INVALID; }
    if (!run || !mm_masters) { set_error("NULL run array or market-maker masters"); return SGMM_ERR_INVALID; }
    if (cfg->use_arl && !adv_masters) { set_error("use_arl needs adversary masters [runs][1250]"); return SGMM_ERR_INVALID; }
    if (cfg->pop_size <= 0) { set_error("pop_size (lambda per run) must be > 0"); return SGMM_ERR_INVALID; }
    if (cfg->shard_stride != 0 || cfg->shard_first != 0 || cfg->shard_count != cfg->pop_size) {
        set_error("a GA sweep runs on one rank: pass an unsharded cfg (shard_first 0, shard_count = pop_size, shard_stride 0)");
        return SGMM_ERR_INVALID;
    }
    if (cfg->max_generations <= 0) { set_error("max_generations must be > 0"); return SGMM_ERR_INVALID; }
    sgmm_ga* ga = new (std::nothrow) sgmm_ga();
    if (!ga) { set_error("out of host memory"); return SGMM_ERR_NOMEM; }
    std::vector<GaDev> init;
    try { init.resize((size_t)runs); } catch (...) { delete ga; set_error("out of host memory"); return SGMM_ERR_NOMEM; }
    for (int32_t r = 0; r < runs; ++r) init[r] = initial_state(run[r].sigma, run[r].patience, run[r].seed, run[r].phi, run[r].fee_rate);
    ga->device = device; ga->cfg = *cfg; ga->G = genome_len(32);
    ga->runs = runs; ga->sweep = true;
    const int64_t P = (int64_t)runs * cfg->pop_size;               // the K*lambda children, one unsharded block
    ga->gather.stride = P; ga->gather.block_bytes = (P * 12 + 15) / 16 * 16;
    ga->capacity = ga->gather.block_bytes;
    if (int rc = ga_allocate(ga, init.data(), mm_masters, adv_masters, (cudaStream_t)stream)) { sgmm_ga_destroy(ga); return rc; }
    *out = ga;
    return SGMM_OK;
}

int sgmm_ga_destroy(sgmm_ga* ga)
{
    if (!ga) return SGMM_OK;
    {
        DeviceGuard guard(ga->device);
        cudaFree(ga->mm_master); cudaFree(ga->adv_master); cudaFree(ga->best_master);
        cudaFree(ga->gather.base); cudaFree(ga->val_fit); cudaFree(ga->val_trd);
        cudaFree(ga->st); cudaFree(ga->h_train_f); cudaFree(ga->h_val_f); cudaFree(ga->h_train_t);
        cudaFree(ga->h_val_t); cudaFree(ga->h_sigma);
        cudaFree(ga->weights); cudaFree(ga->mm_parents); cudaFree(ga->adv_parents);
        es_free(ga);
    }
    delete ga;
    return SGMM_OK;
}

int sgmm_ga_buffers(sgmm_ga* ga, double** fitness_slice, int32_t** trades_slice, void** gather_base,
                    int64_t* block_bytes, int32_t* n_blocks, int32_t* my_block)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    if (ga->runs != 1) { set_error("sgmm_ga_buffers: this GA is a sweep of %d runs on one rank; it has no shard buffers to gather", (int)ga->runs); return SGMM_ERR_INVALID; }
    if (fitness_slice) *fitness_slice = ga->my_fit();
    if (trades_slice) *trades_slice = ga->my_trd();
    if (gather_base) *gather_base = ga->gather.base;
    if (block_bytes) *block_bytes = ga->gather.block_bytes;
    if (n_blocks) *n_blocks = (int32_t)ga->n_blocks;
    if (my_block) *my_block = (int32_t)ga->my_block;
    return SGMM_OK;
}

int sgmm_ga_evaluate(sgmm_ga* ga, const sgmm_bundle* train, void* stream)
{
    if (!ga || !train) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    if (train->device != ga->device) { set_error("bundle and GA live on different devices"); return SGMM_ERR_INVALID; }
    DeviceGuard guard(ga->device);
    ga->started = true;
    const sgmm_ga_config& c = ga->cfg;
    if (ga->sweep) {                                                // run r's children are individuals [r*lambda, (r+1)*lambda)
        const SweepPop mm{ga->mm_master, ga->st, c.pop_size, 0, (int64_t)ga->runs * c.pop_size, 0};
        SweepPop adv = mm;
        adv.master = ga->adv_master; adv.adv = 1;
        return launch_sweep_population(train, mm, c.use_arl ? &adv : nullptr, ga->my_fit(), ga->my_trd(), (cudaStream_t)stream,
                                       ga->objective);
    }
    PopArgs mm{};
    mm.genomes = nullptr; mm.master = ga->mm_master; mm.sigma = c.sigma; mm.sigma_dev = &ga->st->sigma;
    mm.seed = c.seed; mm.generation = 0; mm.generation_dev = &ga->st->generation;
    mm.first_index = c.shard_first; mm.count = c.shard_count; mm.first_index_dev = nullptr;
    PopArgs adv = mm;
    adv.master = ga->adv_master; adv.sigma_dev = &ga->st->adv_sigma; adv.seed = c.seed ^ ADV_SEED_FLIP;
    return launch_population(train, mm, c.use_arl ? &adv : nullptr, c.hidden, c.precision, c.phi, c.fee_rate, 0, 0,
                             ga->my_fit(), ga->my_trd(), (cudaStream_t)stream, ga->objective);
}

int sgmm_ga_select(sgmm_ga* ga, const sgmm_bundle* val, void* stream)
{
    if (!ga || !val) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    if (val->device != ga->device) { set_error("bundle and GA live on different devices"); return SGMM_ERR_INVALID; }
    DeviceGuard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    const sgmm_ga_config& c = ga->cfg;
    ga->started = true;
    if (ga->es_lr > 0.0f) {
        const int64_t lam = c.pop_size;
        es_rank_kernel<<<dim3((unsigned)ga->runs, (unsigned)((lam + ES_RANK_THREADS - 1) / ES_RANK_THREADS)), ES_RANK_THREADS, 0, st>>>(
            ga->st, ga->gather, lam, ga->es_u, ga->es_adv_u, ga->es_pow, c.use_arl);
        if (int rc = check_cuda(cudaGetLastError(), "es_rank_kernel launch")) return rc;
        const int64_t quads = 4 * ES_GRAD_QUADS;
        const int mm_blocks = (int)((ga->G + quads - 1) / quads), adv_blocks = c.use_arl ? (int)((1250 + quads - 1) / quads) : 0;
        es_grad_kernel<<<dim3((unsigned)ga->runs, (unsigned)(mm_blocks + adv_blocks), (unsigned)ga->es_nseg), ES_GRAD_THREADS, 0, st>>>(
            ga->st, lam, ga->es_u, ga->es_adv_u, ga->es_part, ga->es_adv_part, ga->G, mm_blocks);
        if (int rc = check_cuda(cudaGetLastError(), "es_grad_kernel launch")) return rc;
        const int mm_eblocks = (int)((ga->G + ES_ADAM_THREADS - 1) / ES_ADAM_THREADS);
        const int adv_eblocks = c.use_arl ? (1250 + ES_ADAM_THREADS - 1) / ES_ADAM_THREADS : 0;
        es_adam_kernel<<<dim3((unsigned)ga->runs, (unsigned)(mm_eblocks + adv_eblocks)), ES_ADAM_THREADS, 0, st>>>(
            ga->st, lam, ga->es_nseg, ga->es_lr, ga->es_pow, ga->es_part, ga->es_adv_part, ga->es_grad, ga->es_adv_grad,
            ga->es_m, ga->es_adv_m, ga->es_v, ga->es_adv_v, ga->mm_master, ga->adv_master, ga->G, mm_eblocks);
        if (int rc = check_cuda(cudaGetLastError(), "es_adam_kernel launch")) return rc;
    } else if (!ga->weights) {
        ga_tell_kernel<<<(unsigned)ga->runs, 256, 0, st>>>(ga->st, ga->gather, c.pop_size, ga->mm_master, ga->G,
                                                           ga->adv_master, c.use_arl);
        if (int rc = check_cuda(cudaGetLastError(), "ga_tell_kernel launch")) return rc;
    } else {
        ga_select_kernel<<<(unsigned)ga->runs, SELECT_THREADS, 0, st>>>(ga->st, ga->gather, c.pop_size, ga->parents,
                                                                        ga->mm_parents, ga->adv_parents, c.use_arl);
        if (int rc = check_cuda(cudaGetLastError(), "ga_select_kernel launch")) return rc;
        const int64_t quads = RECOMBINE_THREADS * 4;
        const int mm_blocks = (int)((ga->G + quads - 1) / quads), adv_blocks = c.use_arl ? (int)((1250 + quads - 1) / quads) : 0;
        ga_recombine_kernel<<<dim3((unsigned)ga->runs, (unsigned)(mm_blocks + adv_blocks)), RECOMBINE_THREADS, 0, st>>>(
            ga->st, ga->parents, ga->weights, ga->mm_parents, ga->adv_parents, ga->mm_master, ga->G, ga->adv_master, mm_blocks);
        if (int rc = check_cuda(cudaGetLastError(), "ga_recombine_kernel launch")) return rc;
    }
    if (ga->sweep) {                                                // the new masters (best children, or recombined): [runs] rows
        if (int rc = launch_sweep_validation(val, ga->mm_master, ga->st, ga->runs, ga->val_fit, ga->val_trd, st, ga->objective)) return rc;
    } else {
        PopArgs one{};
        one.genomes = ga->mm_master; one.master = nullptr; one.count = 1;      // the new master (best child, or recombined)
        // H = 256: the population's own route (exact, or the same tensor-core path).  H = 32: always exact -- one individual,
        // adversary off, so launch_rollout takes the small-population path of sgmm_one.cu (policy for every (bar, inventory)
        // in parallel, automaton scan, reference-order sum; bit-identical to the sequential kernel)
        const int val_precision = c.hidden == 32 ? SGMM_PRECISION_F32 : c.precision;
        if (int rc = launch_population(val, one, nullptr, c.hidden, val_precision, c.phi, c.fee_rate, 0, 0, ga->val_fit, ga->val_trd, st,
                                       ga->objective)) return rc;
    }
    ga_update_kernel<<<(unsigned)ga->runs, 256, 0, st>>>(ga->st, ga->val_fit, ga->val_trd, ga->mm_master, ga->best_master, ga->G,
                                                         c.use_arl, c.max_generations, ga->h_train_f, ga->h_val_f,
                                                         ga->h_train_t, ga->h_val_t, ga->h_sigma);
    return check_cuda(cudaGetLastError(), "ga_update_kernel launch");
}

int sgmm_ga_generation(sgmm_ga* ga, const sgmm_bundle* train, const sgmm_bundle* val, void* stream)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    if (ga->n_blocks != 1 || ga->cfg.shard_count != ga->cfg.pop_size) {
        set_error("sgmm_ga_generation is the single-rank path; sharded GAs call evaluate / all-gather / select");
        return SGMM_ERR_INVALID;
    }
    if (int rc = sgmm_ga_evaluate(ga, train, stream)) return rc;
    return sgmm_ga_select(ga, val, stream);
}

int sgmm_ga_run_status_host(sgmm_ga* ga, int32_t run, sgmm_ga_status* status, void* stream)
{
    if (!ga || !status) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    if (int rc = check_run(ga, run)) return rc;
    DeviceGuard guard(ga->device);
    GaDev h;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = check_cuda(cudaMemcpyAsync(&h, ga->st + run, sizeof h, cudaMemcpyDeviceToHost, st), "D2H ga state")) return rc;
    if (int rc = check_cuda(cudaStreamSynchronize(st), "ga_status")) return rc;
    status->generation = h.generation; status->stale = h.stale; status->sigma = h.sigma; status->adv_sigma = h.adv_sigma;
    status->best_val = h.best_val; status->last_best_index = h.best_idx;
    return SGMM_OK;
}

int sgmm_ga_run_master_host(sgmm_ga* ga, int32_t run, float* mm_master, float* adv_master, float* best_val_master, void* stream)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    if (int rc = check_run(ga, run)) return rc;
    DeviceGuard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t G = (size_t)ga->G, r = (size_t)run;
    if (mm_master) if (int rc = check_cuda(cudaMemcpyAsync(mm_master, ga->mm_master + r * G, G * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H master")) return rc;
    if (adv_master) if (int rc = check_cuda(cudaMemcpyAsync(adv_master, ga->adv_master + r * 1250, 1250 * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H adv master")) return rc;
    if (best_val_master) if (int rc = check_cuda(cudaMemcpyAsync(best_val_master, ga->best_master + r * G, G * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H best master")) return rc;
    return check_cuda(cudaStreamSynchronize(st), "ga_master");
}

int sgmm_ga_run_history_host(sgmm_ga* ga, int32_t run, int32_t n, double* train_f, double* val_f, int32_t* train_trades,
                             int32_t* val_trades, float* sigma, void* stream)
{
    if (!ga || n < 0) { set_error("bad argument"); return SGMM_ERR_INVALID; }
    if (int rc = check_run(ga, run)) return rc;
    if (n > ga->cfg.max_generations) n = ga->cfg.max_generations;
    DeviceGuard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t k = (size_t)n, row = (size_t)run * (size_t)ga->cfg.max_generations;
    if (train_f) if (int rc = check_cuda(cudaMemcpyAsync(train_f, ga->h_train_f + row, k * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    if (val_f) if (int rc = check_cuda(cudaMemcpyAsync(val_f, ga->h_val_f + row, k * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    if (train_trades) if (int rc = check_cuda(cudaMemcpyAsync(train_trades, ga->h_train_t + row, k * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    if (val_trades) if (int rc = check_cuda(cudaMemcpyAsync(val_trades, ga->h_val_t + row, k * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    if (sigma) if (int rc = check_cuda(cudaMemcpyAsync(sigma, ga->h_sigma + row, k * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    return check_cuda(cudaStreamSynchronize(st), "ga_history");
}

int sgmm_ga_status_host(sgmm_ga* ga, sgmm_ga_status* status, void* stream)
{
    if (!ga || !status) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    if (int rc = single_run(ga, "sgmm_ga_status_host")) return rc;
    return sgmm_ga_run_status_host(ga, 0, status, stream);
}

int sgmm_ga_master_host(sgmm_ga* ga, float* mm_master, float* adv_master, float* best_val_master, void* stream)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    if (int rc = single_run(ga, "sgmm_ga_master_host")) return rc;
    return sgmm_ga_run_master_host(ga, 0, mm_master, adv_master, best_val_master, stream);
}

int sgmm_ga_history_host(sgmm_ga* ga, int32_t n, double* train_f, double* val_f, int32_t* train_trades,
                         int32_t* val_trades, float* sigma, void* stream)
{
    if (!ga || n < 0) { set_error("bad argument"); return SGMM_ERR_INVALID; }
    if (int rc = single_run(ga, "sgmm_ga_history_host")) return rc;
    return sgmm_ga_run_history_host(ga, 0, n, train_f, val_f, train_trades, val_trades, sigma, stream);
}

int sgmm_ga_set_parents(sgmm_ga* ga, int32_t parents, const float* weights, void* stream)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    if (ga->started) {
        set_error("sgmm_ga_set_parents: a generation of this GA has already been enqueued; set the parents right after create");
        return SGMM_ERR_INVALID;
    }
    if (ga->es_lr > 0.0f) {
        set_error("sgmm_ga_set_parents: this GA runs the evolution strategy (sgmm_ga_set_es); the two updates exclude each other");
        return SGMM_ERR_INVALID;
    }
    if (parents < 1 || parents > SGMM_MAX_PARENTS || parents > ga->cfg.pop_size) {
        set_error("parents=%d: need 1 <= parents <= min(pop_size=%lld, %d)", (int)parents, (long long)ga->cfg.pop_size,
                  SGMM_MAX_PARENTS);
        return SGMM_ERR_INVALID;
    }
    std::vector<float> w((size_t)parents, 1.0f / (float)parents);
    if (weights) {
        bool any = false;
        for (int32_t k = 0; k < parents; ++k) {
            if (!std::isfinite(weights[k]) || weights[k] < 0.0f) { set_error("weight %d = %g: weights must be finite and >= 0", (int)k, (double)weights[k]); return SGMM_ERR_INVALID; }
            any = any || weights[k] > 0.0f;
            w[k] = weights[k];
        }
        if (!any) { set_error("every recombination weight is 0"); return SGMM_ERR_INVALID; }
    }
    DeviceGuard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    cudaFree(ga->weights); cudaFree(ga->mm_parents); cudaFree(ga->adv_parents);     // a second call before the first generation
    ga->weights = nullptr; ga->mm_parents = ga->adv_parents = nullptr;
    const size_t n = (size_t)ga->runs * (size_t)parents;
    int rc = SGMM_OK;
    if (!rc) rc = check_cuda(cudaMalloc(&ga->mm_parents, n * sizeof(int64_t)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->adv_parents, n * sizeof(int64_t)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->weights, (size_t)parents * sizeof(float)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->mm_parents, 0, n * sizeof(int64_t), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->adv_parents, 0, n * sizeof(int64_t), st), "memset");
    if (!rc) rc = check_cuda(cudaMemcpyAsync(ga->weights, w.data(), (size_t)parents * sizeof(float), cudaMemcpyHostToDevice, st), "H2D weights");
    if (!rc) rc = check_cuda(cudaStreamSynchronize(st), "ga_set_parents");
    if (rc) {                                                       // back to the (1,lambda) GA
        cudaFree(ga->weights); cudaFree(ga->mm_parents); cudaFree(ga->adv_parents);
        ga->weights = nullptr; ga->mm_parents = ga->adv_parents = nullptr;
        return rc;
    }
    ga->parents = parents;
    return SGMM_OK;
}

int sgmm_ga_run_parents_host(sgmm_ga* ga, int32_t run, int32_t n, int64_t* mm_index, int64_t* adv_index, void* stream)
{
    if (!ga || n < 0) { set_error("bad argument"); return SGMM_ERR_INVALID; }
    if (int rc = check_run(ga, run)) return rc;
    const size_t k = (size_t)(n < ga->parents ? n : ga->parents), r = (size_t)run;
    if (k == 0) return SGMM_OK;
    DeviceGuard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (!ga->weights) {                                             // (1,lambda): the best children of the state
        GaDev h;
        if (int rc = check_cuda(cudaMemcpyAsync(&h, ga->st + run, sizeof h, cudaMemcpyDeviceToHost, st), "D2H ga state")) return rc;
        if (int rc = check_cuda(cudaStreamSynchronize(st), "ga_parents")) return rc;
        if (mm_index) mm_index[0] = h.best_idx;
        if (adv_index) adv_index[0] = h.adv_best_idx;
        return SGMM_OK;
    }
    const size_t P = (size_t)ga->parents;
    if (mm_index) if (int rc = check_cuda(cudaMemcpyAsync(mm_index, ga->mm_parents + r * P, k * sizeof(int64_t), cudaMemcpyDeviceToHost, st), "D2H parents")) return rc;
    if (adv_index) if (int rc = check_cuda(cudaMemcpyAsync(adv_index, ga->adv_parents + r * P, k * sizeof(int64_t), cudaMemcpyDeviceToHost, st), "D2H parents")) return rc;
    return check_cuda(cudaStreamSynchronize(st), "ga_parents");
}

int sgmm_ga_parents_host(sgmm_ga* ga, int32_t n, int64_t* mm_index, int64_t* adv_index, void* stream)
{
    if (!ga || n < 0) { set_error("bad argument"); return SGMM_ERR_INVALID; }
    if (int rc = single_run(ga, "sgmm_ga_parents_host")) return rc;
    return sgmm_ga_run_parents_host(ga, 0, n, mm_index, adv_index, stream);
}

int sgmm_ga_set_es(sgmm_ga* ga, float lr, void* stream)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    if (ga->started) {
        set_error("sgmm_ga_set_es: a generation of this GA has already been enqueued; set the evolution strategy right after create");
        return SGMM_ERR_INVALID;
    }
    if (!std::isfinite(lr) || !(lr > 0.0f)) { set_error("lr=%g: the Adam step size must be finite and > 0", (double)lr); return SGMM_ERR_INVALID; }
    if (ga->weights) {
        set_error("sgmm_ga_set_es: this GA runs truncation selection (sgmm_ga_set_parents); the two updates exclude each other");
        return SGMM_ERR_INVALID;
    }
    const int64_t lam = ga->cfg.pop_size;
    if (lam < 2) { set_error("pop_size=%lld: centered-rank utilities need lambda >= 2", (long long)lam); return SGMM_ERR_INVALID; }
    if (lam > (int64_t)65535 * ES_RANK_THREADS) {
        set_error("pop_size=%lld: the evolution strategy ranks at most %lld children per run", (long long)lam,
                  (long long)65535 * ES_RANK_THREADS);
        return SGMM_ERR_INVALID;
    }
    DeviceGuard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    es_free(ga);                                                    // a second call before the first generation
    const size_t R = (size_t)ga->runs, G = (size_t)ga->G, L = (size_t)lam, S = (size_t)((lam + ES_SEGMENT - 1) / ES_SEGMENT);
    struct { float** p; size_t n; } bufs[] = {
        {&ga->es_u, R * L}, {&ga->es_adv_u, R * L}, {&ga->es_part, R * S * G}, {&ga->es_adv_part, R * S * 1250},
        {&ga->es_grad, R * G}, {&ga->es_adv_grad, R * 1250}, {&ga->es_m, R * G}, {&ga->es_adv_m, R * 1250},
        {&ga->es_v, R * G}, {&ga->es_adv_v, R * 1250}, {&ga->es_pow, R * 2}};
    int rc = SGMM_OK;
    for (auto& b : bufs) {
        if (!rc) rc = check_cuda(cudaMalloc(b.p, b.n * sizeof(float)), "cudaMalloc");
        if (!rc) rc = check_cuda(cudaMemsetAsync(*b.p, 0, b.n * sizeof(float), st), "memset");
    }
    std::vector<float> ones(2 * R, 1.0f);                           // b1^0, b2^0
    if (!rc) rc = check_cuda(cudaMemcpyAsync(ga->es_pow, ones.data(), 2 * R * sizeof(float), cudaMemcpyHostToDevice, st), "H2D es powers");
    if (!rc) rc = check_cuda(cudaStreamSynchronize(st), "ga_set_es");
    if (rc) { es_free(ga); return rc; }                             // back to the (1,lambda) GA
    ga->es_lr = lr; ga->es_nseg = (int32_t)S;
    return SGMM_OK;
}

int sgmm_ga_set_objective(sgmm_ga* ga, int32_t objective, void* stream)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    if (ga->started) {
        set_error("sgmm_ga_set_objective: a generation of this GA has already been enqueued; set the objective right after create");
        return SGMM_ERR_INVALID;
    }
    if (objective < SGMM_OBJECTIVE_REWARD || objective > SGMM_OBJECTIVE_SHARPE) { set_error("unknown objective %d", (int)objective); return SGMM_ERR_INVALID; }
    const int p = ga->cfg.precision;
    if (objective != SGMM_OBJECTIVE_REWARD && p != SGMM_PRECISION_F32 && p != SGMM_PRECISION_EXACT) {
        set_error("objective %d: training objectives run in SGMM-F32 order only; this GA has the tensor-core precision %d "
                  "(create it with SGMM_PRECISION_EXACT)", (int)objective, p);
        return SGMM_ERR_UNSUPPORTED;
    }
    DeviceGuard guard(ga->device);
    if (int rc = check_cuda(cudaStreamSynchronize((cudaStream_t)stream), "ga_set_objective")) return rc;
    ga->objective = objective;
    return SGMM_OK;
}

int sgmm_ga_run_es_host(sgmm_ga* ga, int32_t run, float* utilities, float* grad, float* adv_utilities, float* adv_grad,
                        void* stream)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    if (int rc = check_run(ga, run)) return rc;
    if (!(ga->es_lr > 0.0f)) { set_error("sgmm_ga_run_es_host: this GA does not run the evolution strategy (sgmm_ga_set_es)"); return SGMM_ERR_INVALID; }
    DeviceGuard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t L = (size_t)ga->cfg.pop_size, G = (size_t)ga->G, r = (size_t)run;
    if (utilities) if (int rc = check_cuda(cudaMemcpyAsync(utilities, ga->es_u + r * L, L * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H es")) return rc;
    if (grad) if (int rc = check_cuda(cudaMemcpyAsync(grad, ga->es_grad + r * G, G * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H es")) return rc;
    if (adv_utilities) if (int rc = check_cuda(cudaMemcpyAsync(adv_utilities, ga->es_adv_u + r * L, L * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H es")) return rc;
    if (adv_grad) if (int rc = check_cuda(cudaMemcpyAsync(adv_grad, ga->es_adv_grad + r * 1250, 1250 * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H es")) return rc;
    return check_cuda(cudaStreamSynchronize(st), "ga_es");
}

int sgmm_ga_es_host(sgmm_ga* ga, float* utilities, float* grad, float* adv_utilities, float* adv_grad, void* stream)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    if (int rc = single_run(ga, "sgmm_ga_es_host")) return rc;
    return sgmm_ga_run_es_host(ga, 0, utilities, grad, adv_utilities, adv_grad, stream);
}

}  // extern "C"
