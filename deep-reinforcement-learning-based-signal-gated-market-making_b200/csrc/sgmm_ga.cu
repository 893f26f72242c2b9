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
#include <new>
#include "sgmm_internal.h"
#include "sgmm_rng.cuh"

namespace sgmm {

struct GaDev {
    int32_t generation;
    int32_t stale;
    float sigma, adv_sigma;
    double best_val;
    int64_t best_idx, adv_best_idx;
    double train_f; int32_t train_trades; int32_t pad;
};

constexpr uint64_t ADV_SEED_FLIP = 0x8000000000000000ull;   // adversary noise stream (same as the oracle)

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

// numpy argmax over fitness (SIGN=+1) or over -fitness (SIGN=-1): first maximum, first NaN wins
template <int SIGN>
__device__ int64_t block_argmax(const Gather& f, int64_t n, double* s_val, int64_t* s_idx)
{
    const int tid = threadIdx.x, nt = blockDim.x;
    double bv = 0.0; int64_t bi = -1; bool bnan = false;
    for (int64_t i = tid; i < n; i += nt) {
        const double v = SIGN > 0 ? f.fit(i) : -f.fit(i);
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

__global__ void __launch_bounds__(256) ga_tell_kernel(GaDev* st, const Gather fit, int64_t pop,
                                                      float* mm_master, int64_t G, float* adv_master, int use_arl,
                                                      uint64_t seed)
{
    __shared__ double s_val[256];
    __shared__ int64_t s_idx[256];
    const int64_t best = block_argmax<+1>(fit, pop, s_val, s_idx);
    int64_t abest = 0;
    if (use_arl) abest = block_argmax<-1>(fit, pop, s_val, s_idx);
    const uint64_t gen = (uint64_t)st->generation;
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
        st->train_f = fit.fit(best); st->train_trades = fit.trd(best);
    }
}

__global__ void __launch_bounds__(256) ga_update_kernel(GaDev* st, const double* val_f, const int32_t* val_t,
                                                        const float* mm_master, float* best_master, int64_t G,
                                                        int patience, int use_arl, int max_gen,
                                                        double* h_train_f, double* h_val_f, int32_t* h_train_t,
                                                        int32_t* h_val_t, float* h_sigma)
{
    __shared__ int improved;
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
            h_train_f[g] = st->train_f; h_val_f[g] = *val_f; h_train_t[g] = st->train_trades; h_val_t[g] = *val_t;
            h_sigma[g] = st->sigma;
        }
        if (improved) { st->best_val = *val_f; st->stale = 0; } else st->stale += 1;     // :145-152
        if (st->stale >= patience) {                                // :155-160
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
    int64_t G = 0, capacity = 0;
    float* mm_master = nullptr; float* adv_master = nullptr; float* best_master = nullptr;
    sgmm::Gather gather{nullptr, 0, 0}; int64_t n_blocks = 1, my_block = 0;
    double* my_fit() const { return gather.fit_block(my_block); }          // this rank's slice: children [shard_first, +shard_count)
    int32_t* my_trd() const { return gather.trd_block(my_block); }
    double* val_fit = nullptr; int32_t* val_trd = nullptr;
    GaDev* st = nullptr;
    double* h_train_f = nullptr; double* h_val_f = nullptr; int32_t* h_train_t = nullptr; int32_t* h_val_t = nullptr;
    float* h_sigma = nullptr;
};

namespace {
struct Guard {
    int prev = -1;
    explicit Guard(int d) { cudaGetDevice(&prev); cudaSetDevice(d); }
    ~Guard() { if (prev >= 0) cudaSetDevice(prev); }
};
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
    Guard guard(device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t G = (size_t)ga->G, cap = (size_t)ga->capacity, mg = (size_t)cfg->max_generations;
    int rc = SGMM_OK;
    if (!rc) rc = check_cuda(cudaMalloc(&ga->mm_master, G * sizeof(float)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->best_master, G * sizeof(float)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->adv_master, 1250 * sizeof(float)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->gather.base, cap), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->val_fit, sizeof(double)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->val_trd, sizeof(int32_t)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->st, sizeof(GaDev)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_train_f, mg * sizeof(double)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_val_f, mg * sizeof(double)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_train_t, mg * sizeof(int32_t)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_val_t, mg * sizeof(int32_t)), "cudaMalloc");
    if (!rc) rc = check_cuda(cudaMalloc(&ga->h_sigma, mg * sizeof(float)), "cudaMalloc");
    GaDev init{};
    init.generation = 0; init.stale = 0; init.sigma = cfg->sigma; init.adv_sigma = cfg->sigma;
    init.best_val = -INFINITY;                                      // drl_engine.py:84
    if (!rc) rc = check_cuda(cudaMemcpyAsync(ga->st, &init, sizeof init, cudaMemcpyHostToDevice, st), "H2D ga state");
    if (!rc) rc = check_cuda(cudaMemcpyAsync(ga->mm_master, mm_master, G * sizeof(float), cudaMemcpyHostToDevice, st), "H2D master");
    if (!rc) rc = check_cuda(cudaMemcpyAsync(ga->best_master, mm_master, G * sizeof(float), cudaMemcpyHostToDevice, st), "H2D master");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->adv_master, 0, 1250 * sizeof(float), st), "memset");
    if (!rc && adv_master) rc = check_cuda(cudaMemcpyAsync(ga->adv_master, adv_master, 1250 * sizeof(float), cudaMemcpyHostToDevice, st), "H2D adv master");
    // history of generations not yet run reads as zeros (sgmm_ga_history_host additionally clamps n to the generations completed)
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_train_f, 0, mg * sizeof(double), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_val_f, 0, mg * sizeof(double), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_train_t, 0, mg * sizeof(int32_t), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_val_t, 0, mg * sizeof(int32_t), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->h_sigma, 0, mg * sizeof(float), st), "memset");
    if (!rc) rc = check_cuda(cudaMemsetAsync(ga->gather.base, 0, cap, st), "memset");
    if (!rc) rc = check_cuda(cudaStreamSynchronize(st), "ga_create");
    if (rc) { sgmm_ga_destroy(ga); return rc; }
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
    ga_tell_kernel<<<1, 256, 0, st>>>(ga->st, ga->gather, c.pop_size, ga->mm_master, ga->G,
                                      ga->adv_master, c.use_arl, c.seed);
    if (int rc = check_cuda(cudaGetLastError(), "ga_tell_kernel launch")) return rc;
    PopArgs one{};
    one.genomes = ga->mm_master; one.master = nullptr; one.count = 1;          // the new master IS the best child
    // H = 256: the population's own route (exact, or the same tensor-core path).  H = 32: always exact -- one individual,
    // adversary off, so launch_rollout takes the small-population path of sgmm_one.cu (policy for every (bar, inventory)
    // in parallel, automaton scan, reference-order sum; bit-identical to the sequential kernel)
    const int val_precision = c.hidden == 32 ? SGMM_PRECISION_F32 : c.precision;
    if (int rc = launch_population(val, one, nullptr, c.hidden, val_precision, c.phi, c.fee_rate, 0, 0, ga->val_fit, ga->val_trd, st)) return rc;
    ga_update_kernel<<<1, 256, 0, st>>>(ga->st, ga->val_fit, ga->val_trd, ga->mm_master, ga->best_master, ga->G,
                                        c.patience, c.use_arl, c.max_generations, ga->h_train_f, ga->h_val_f,
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

int sgmm_ga_status_host(sgmm_ga* ga, sgmm_ga_status* status, void* stream)
{
    if (!ga || !status) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    Guard guard(ga->device);
    GaDev h;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = check_cuda(cudaMemcpyAsync(&h, ga->st, sizeof h, cudaMemcpyDeviceToHost, st), "D2H ga state")) return rc;
    if (int rc = check_cuda(cudaStreamSynchronize(st), "ga_status")) return rc;
    status->generation = h.generation; status->stale = h.stale; status->sigma = h.sigma; status->adv_sigma = h.adv_sigma;
    status->best_val = h.best_val; status->last_best_index = h.best_idx;
    return SGMM_OK;
}

int sgmm_ga_master_host(sgmm_ga* ga, float* mm_master, float* adv_master, float* best_val_master, void* stream)
{
    if (!ga) { set_error("ga is NULL"); return SGMM_ERR_INVALID; }
    Guard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t G = (size_t)ga->G;
    if (mm_master) if (int rc = check_cuda(cudaMemcpyAsync(mm_master, ga->mm_master, G * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H master")) return rc;
    if (adv_master) if (int rc = check_cuda(cudaMemcpyAsync(adv_master, ga->adv_master, 1250 * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H adv master")) return rc;
    if (best_val_master) if (int rc = check_cuda(cudaMemcpyAsync(best_val_master, ga->best_master, G * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H best master")) return rc;
    return check_cuda(cudaStreamSynchronize(st), "ga_master");
}

int sgmm_ga_history_host(sgmm_ga* ga, int32_t n, double* train_f, double* val_f, int32_t* train_trades,
                         int32_t* val_trades, float* sigma, void* stream)
{
    if (!ga || n < 0) { set_error("bad argument"); return SGMM_ERR_INVALID; }
    if (n > ga->cfg.max_generations) n = ga->cfg.max_generations;
    Guard guard(ga->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t k = (size_t)n;
    if (train_f) if (int rc = check_cuda(cudaMemcpyAsync(train_f, ga->h_train_f, k * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    if (val_f) if (int rc = check_cuda(cudaMemcpyAsync(val_f, ga->h_val_f, k * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    if (train_trades) if (int rc = check_cuda(cudaMemcpyAsync(train_trades, ga->h_train_t, k * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    if (val_trades) if (int rc = check_cuda(cudaMemcpyAsync(val_trades, ga->h_val_t, k * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    if (sigma) if (int rc = check_cuda(cudaMemcpyAsync(sigma, ga->h_sigma, k * sizeof(float), cudaMemcpyDeviceToHost, st), "D2H history")) return rc;
    return check_cuda(cudaStreamSynchronize(st), "ga_history");
}

}  // extern "C"
