// sgmm_ga.cu -- device-side (1,lambda) evolution: NeuroEvolution.ask/tell and the generation loop
// of DRLEngine.train (/root/reference/models/model.py:59-76, Env/drl_engine.py:92-171) with no
// host round trip inside a generation.
//   ask       children are never materialised: the rollout kernel regenerates child i from
//             (master, sigma, seed, generation, i) with the counter-based noise of sgmm_rng.cuh
//   tell      argmax with numpy's semantics (first maximum, a NaN wins) -> master <- that child
//             (model.py:73-76); the adversary is told -fitness (drl_engine.py:123-125)
//   validate  rollout of the new master (== best child, drl_engine.py:129-140) with no adversary
//   select    keep-best-on-validation snapshot (:144-150), sigma halving after `patience` stale
//             generations (:155-160), history (:163-167)
// A sweep (sgmm_ga_create_sweep) advances K independent runs with the same launches: K*lambda children in one policy
// table and one walk (sgmm_one.cu), one tell block and one update block per run, the K new masters validated as one
// population.  Each run's state is its own GaDev (sgmm_internal.h) and history row; run r is bit-identical to the solo GA
// of its seed, phi, fee, sigma and patience.  A GA from sgmm_ga_create is the one-run case of the same kernels.
#include <new>
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
};

namespace {
struct Guard {
    int prev = -1;
    explicit Guard(int d) { cudaGetDevice(&prev); cudaSetDevice(d); }
    ~Guard() { if (prev >= 0) cudaSetDevice(prev); }
};

// device buffers of ga->runs runs, initial states `init` [runs] and HOST masters [runs][G] / [runs][1250] (adv may be NULL)
int ga_allocate(sgmm_ga* ga, const GaDev* init, const float* mm_masters, const float* adv_masters, cudaStream_t st)
{
    Guard guard(ga->device);
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
        Guard guard(ga->device);
        cudaFree(ga->mm_master); cudaFree(ga->adv_master); cudaFree(ga->best_master);
        cudaFree(ga->gather.base); cudaFree(ga->val_fit); cudaFree(ga->val_trd);
        cudaFree(ga->st); cudaFree(ga->h_train_f); cudaFree(ga->h_val_f); cudaFree(ga->h_train_t);
        cudaFree(ga->h_val_t); cudaFree(ga->h_sigma);
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
    Guard guard(ga->device);
    const sgmm_ga_config& c = ga->cfg;
    if (ga->sweep) {                                                // run r's children are individuals [r*lambda, (r+1)*lambda)
        const SweepPop mm{ga->mm_master, ga->st, c.pop_size, 0, (int64_t)ga->runs * c.pop_size, 0};
        SweepPop adv = mm;
        adv.master = ga->adv_master; adv.adv = 1;
        return launch_sweep_population(train, mm, c.use_arl ? &adv : nullptr, ga->my_fit(), ga->my_trd(), (cudaStream_t)stream);
    }
    PopArgs mm{};
    mm.genomes = nullptr; mm.master = ga->mm_master; mm.sigma = c.sigma; mm.sigma_dev = &ga->st->sigma;
    mm.seed = c.seed; mm.generation = 0; mm.generation_dev = &ga->st->generation;
    mm.first_index = c.shard_first; mm.count = c.shard_count; mm.first_index_dev = nullptr;
    PopArgs adv = mm;
    adv.master = ga->adv_master; adv.sigma_dev = &ga->st->adv_sigma; adv.seed = c.seed ^ ADV_SEED_FLIP;
    return launch_population(train, mm, c.use_arl ? &adv : nullptr, c.hidden, c.precision, c.phi, c.fee_rate, 0, 0,
                             ga->my_fit(), ga->my_trd(), (cudaStream_t)stream);
}

int sgmm_ga_select(sgmm_ga* ga, const sgmm_bundle* val, void* stream)
{
    if (!ga || !val) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    if (val->device != ga->device) { set_error("bundle and GA live on different devices"); return SGMM_ERR_INVALID; }
    Guard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    const sgmm_ga_config& c = ga->cfg;
    ga_tell_kernel<<<(unsigned)ga->runs, 256, 0, st>>>(ga->st, ga->gather, c.pop_size, ga->mm_master, ga->G,
                                                       ga->adv_master, c.use_arl);
    if (int rc = check_cuda(cudaGetLastError(), "ga_tell_kernel launch")) return rc;
    if (ga->sweep) {                                                // the new masters ARE the best children: [runs][1250] rows
        if (int rc = launch_sweep_validation(val, ga->mm_master, ga->st, ga->runs, ga->val_fit, ga->val_trd, st)) return rc;
    } else {
        PopArgs one{};
        one.genomes = ga->mm_master; one.master = nullptr; one.count = 1;      // the new master IS the best child
        // H = 256: the population's own route (exact, or the same tensor-core path).  H = 32: always exact -- one individual,
        // adversary off, so launch_rollout takes the small-population path of sgmm_one.cu (policy for every (bar, inventory)
        // in parallel, automaton scan, reference-order sum; bit-identical to the sequential kernel)
        const int val_precision = c.hidden == 32 ? SGMM_PRECISION_F32 : c.precision;
        if (int rc = launch_population(val, one, nullptr, c.hidden, val_precision, c.phi, c.fee_rate, 0, 0, ga->val_fit, ga->val_trd, st)) return rc;
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
    Guard guard(ga->device);
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
    Guard guard(ga->device);
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
    Guard guard(ga->device);
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

}  // extern "C"
