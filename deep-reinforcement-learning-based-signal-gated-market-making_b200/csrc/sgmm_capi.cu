// sgmm_capi.cu -- the C ABI of include/sgmm.h: handles, argument checking, host<->device staging.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <new>
#include "sgmm_internal.h"
#include "sgmm_step_core.h"

namespace sgmm {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...)
{
    va_list ap; va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

int check_cuda(cudaError_t e, const char* what)
{
    if (e == cudaSuccess) return SGMM_OK;
    set_error("%s: %s", what, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? SGMM_ERR_NOMEM : SGMM_ERR_CUDA;
}

struct DeviceGuard {
    int prev = -1; bool ok = false;
    explicit DeviceGuard(int dev) { if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess) ok = true; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

static int ensure_workspace(sgmm_bundle* b, int slot, size_t bytes)
{
    if (b->ws_bytes[slot] >= bytes) return SGMM_OK;
    if (b->ws[slot]) { cudaFree(b->ws[slot]); b->ws[slot] = nullptr; b->ws_bytes[slot] = 0; }   // cudaFree synchronises: no user left
    size_t want = bytes + bytes / 4 + 4096;
    if (int rc = check_cuda(cudaMalloc(&b->ws[slot], want), "cudaMalloc(workspace)")) return rc;
    b->ws_bytes[slot] = want;
    return SGMM_OK;
}

static int fill_pop(const sgmm_population* p, const char* name, PopArgs& out)
{
    if (p->count < 0) { set_error("%s.count < 0", name); return SGMM_ERR_INVALID; }
    if (p->count > 0 && !p->genomes && !p->master) { set_error("%s: neither genomes nor master given", name); return SGMM_ERR_INVALID; }
    out.genomes = p->genomes; out.master = p->master; out.first_index_dev = nullptr;
    out.sigma = p->sigma; out.sigma_dev = nullptr; out.seed = p->seed; out.generation = p->generation;
    out.generation_dev = nullptr; out.first_index = p->first_index; out.count = p->count;
    return SGMM_OK;
}

static int tc32_mode_of(int precision) { return precision == SGMM_PRECISION_TF32 ? 1 : (precision == SGMM_PRECISION_F16 ? 2 : 0); }

int launch_population(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, int hidden, int precision, double phi, double fee,
                      int units_per_lane, int warps_per_cta, double* fitness, int32_t* trades, cudaStream_t st)
{
    if (precision == SGMM_PRECISION_EXACT && hidden == 32) precision = SGMM_PRECISION_F32;     // EXACT at H = 32 is the F32 route
    if (hidden == 256 && precision == SGMM_PRECISION_EXACT)         // bit-exact H = 256: policy tables + walks, in batches
        return launch_exact256(b, mm, adv, phi, fee, fitness, trades, st);
    if (hidden == 256 && adv && precision == SGMM_PRECISION_BF16)   // spec256 q tables + walk_account_kernel<Walk20>, in batches
        return launch_spec256_adv(b, mm, *adv, phi, fee, fitness, trades, nullptr, nullptr, st);
    if (hidden == 256)                                              // BASELINE config 4: spec256_kernel + account_kernel
        return launch_spec256(b, mm, phi, fee, fitness, trades, nullptr, nullptr, st);
    if (precision != SGMM_PRECISION_F32)                            // tensor cores at H = 32
        return launch_tc32(b, mm, adv, phi, fee, units_per_lane, fitness, trades, nullptr, nullptr, st, tc32_mode_of(precision));
    return launch_rollout(b, mm, adv, hidden, phi, fee, units_per_lane, warps_per_cta, fitness, trades, st);
}

}  // namespace sgmm

using namespace sgmm;

extern "C" {

int sgmm_version(void) { return SGMM_VERSION; }
const char* sgmm_last_error(void) { return g_err; }

int sgmm_abi_sizeof(int which)
{
    switch (which) {
        case 0: return (int)sizeof(sgmm_population);
        case 1: return (int)sizeof(sgmm_rollout_params);
        case 2: return (int)sizeof(sgmm_trace);
        case 3: return (int)sizeof(sgmm_env_state);
        case 4: return (int)sizeof(sgmm_step_info);
        case 5: return (int)sizeof(sgmm_ga_config);
        case 6: return (int)sizeof(sgmm_ga_status);
        default: return SGMM_ERR_INVALID;
    }
}

int sgmm_device_count(void)
{
    int n = 0;
    if (int rc = check_cuda(cudaGetDeviceCount(&n), "cudaGetDeviceCount")) return rc;
    return n;
}

int sgmm_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, uint64_t* total_mem)
{
    cudaDeviceProp p;
    if (int rc = check_cuda(cudaGetDeviceProperties(&p, device), "cudaGetDeviceProperties")) return rc;
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (total_mem) *total_mem = (uint64_t)p.totalGlobalMem;
    return SGMM_OK;
}

int sgmm_bundle_create(sgmm_bundle** out, int64_t T, const float* z1, const float* z2,
                       const double* mid_next, const double* best_ask, const double* best_bid,
                       const double* buy_max, const double* sell_min, double tick_size,
                       int device, void* stream)
{
    if (!out) { set_error("out is NULL"); return SGMM_ERR_INVALID; }
    *out = nullptr;
    if (T < 0) { set_error("T < 0"); return SGMM_ERR_INVALID; }
    if (T > 0 && (!z1 || !z2 || !mid_next || !best_ask || !best_bid || !buy_max || !sell_min)) {
        set_error("NULL bar array with T > 0"); return SGMM_ERR_INVALID;
    }
    if (!(tick_size > 0.0) || !std::isfinite(tick_size)) {
        set_error("tick_size must be finite and > 0 (fill thresholds rely on the quote being monotone in the offset)");
        return SGMM_ERR_INVALID;
    }
    DeviceGuard guard(device);
    if (!guard.ok) { set_error("cannot select CUDA device %d: %s", device, cudaGetErrorString(cudaGetLastError())); return SGMM_ERR_CUDA; }
    cudaDeviceProp prop;
    if (int rc = check_cuda(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties")) return rc;
    if (prop.major != 10) { set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor); return SGMM_ERR_UNSUPPORTED; }
    sgmm_bundle* b = new (std::nothrow) sgmm_bundle();
    if (!b) { set_error("out of host memory"); return SGMM_ERR_NOMEM; }
    b->device = device; b->T = T; b->tick = tick_size;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = SGMM_OK;
    float* dz = nullptr; double* dd = nullptr;
    if (T > 0) {
        const size_t n = (size_t)T;
        if (!rc) rc = check_cuda(cudaMalloc(&b->sig, n * sizeof(BarSig)), "cudaMalloc(sig)");
        if (!rc) rc = check_cuda(cudaMalloc(&b->px, n * sizeof(BarPx)), "cudaMalloc(px)");
        if (!rc) rc = check_cuda(cudaMalloc(&b->bmax, n * sizeof(double)), "cudaMalloc(buy_max)");
        if (!rc) rc = check_cuda(cudaMalloc(&b->smin, n * sizeof(double)), "cudaMalloc(sell_min)");
        if (!rc) rc = check_cuda(cudaMalloc(&b->a1, tc32_a1_bytes(T)), "cudaMalloc(a1 tiles)");
        if (!rc) rc = check_cuda(cudaMalloc(&dz, 2 * n * sizeof(float)), "cudaMalloc(z staging)");
        if (!rc) rc = check_cuda(cudaMalloc(&dd, 3 * n * sizeof(double)), "cudaMalloc(price staging)");
        if (!rc) rc = check_cuda(cudaMemcpyAsync(dz, z1, n * sizeof(float), cudaMemcpyHostToDevice, st), "H2D z1");
        if (!rc) rc = check_cuda(cudaMemcpyAsync(dz + n, z2, n * sizeof(float), cudaMemcpyHostToDevice, st), "H2D z2");
        if (!rc) rc = check_cuda(cudaMemcpyAsync(dd, mid_next, n * sizeof(double), cudaMemcpyHostToDevice, st), "H2D mid_next");
        if (!rc) rc = check_cuda(cudaMemcpyAsync(dd + n, best_ask, n * sizeof(double), cudaMemcpyHostToDevice, st), "H2D best_ask");
        if (!rc) rc = check_cuda(cudaMemcpyAsync(dd + 2 * n, best_bid, n * sizeof(double), cudaMemcpyHostToDevice, st), "H2D best_bid");
        if (!rc) rc = check_cuda(cudaMemcpyAsync(b->bmax, buy_max, n * sizeof(double), cudaMemcpyHostToDevice, st), "H2D buy_max");
        if (!rc) rc = check_cuda(cudaMemcpyAsync(b->smin, sell_min, n * sizeof(double), cudaMemcpyHostToDevice, st), "H2D sell_min");
        if (!rc) rc = launch_prologue(b, dz, dz + n, dd, dd + n, dd + 2 * n, st);
        if (!rc) rc = launch_tc32_prologue(b, st);
        if (!rc) rc = check_cuda(cudaStreamSynchronize(st), "bundle prologue");
        cudaFree(dz); cudaFree(dd);
    }
    if (rc) { sgmm_bundle_destroy(b); return rc; }
    *out = b;
    return SGMM_OK;
}

int sgmm_bundle_length(const sgmm_bundle* b, int64_t* T)
{
    if (!b || !T) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    *T = b->T; return SGMM_OK;
}

int sgmm_bundle_device(const sgmm_bundle* b, int* device)
{
    if (!b || !device) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    *device = b->device; return SGMM_OK;
}

int sgmm_bundle_thresholds(const sgmm_bundle* b, int32_t* ka, int32_t* kb, void* stream)
{
    if (!b) { set_error("bundle is NULL"); return SGMM_ERR_INVALID; }
    if (b->T == 0) return SGMM_OK;
    DeviceGuard guard(b->device);
    BarSig* h = (BarSig*)malloc((size_t)b->T * sizeof(BarSig));
    if (!h) { set_error("out of host memory"); return SGMM_ERR_NOMEM; }
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_cuda(cudaMemcpyAsync(h, b->sig, (size_t)b->T * sizeof(BarSig), cudaMemcpyDeviceToHost, st), "D2H thresholds");
    if (!rc) rc = check_cuda(cudaStreamSynchronize(st), "D2H thresholds");
    if (!rc) for (int64_t t = 0; t < b->T; ++t) {
        // stored as threshold+1 (strict compare); report the threshold itself, sentinels unchanged
        if (ka) ka[t] = (h[t].ka1 == K_NEVER || h[t].ka1 == K_ALWAYS) ? h[t].ka1 : h[t].ka1 - 1;
        if (kb) kb[t] = (h[t].kb1 == K_NEVER || h[t].kb1 == K_ALWAYS) ? h[t].kb1 : h[t].kb1 - 1;
    }
    free(h);
    return rc;
}

int sgmm_bundle_destroy(sgmm_bundle* b)
{
    if (!b) return SGMM_OK;
    {
        DeviceGuard guard(b->device);
        cudaFree(b->sig); cudaFree(b->px); cudaFree(b->bmax); cudaFree(b->smin); cudaFree(b->a1); cudaFree(b->codes);
        for (int k = 0; k < SGMM_HOST_SLOTS; ++k) { if (b->slot_stream[k]) { cudaStreamSynchronize(b->slot_stream[k]); cudaStreamDestroy(b->slot_stream[k]); } cudaFree(b->ws[k]); }
        for (uint64_t* p : b->codes_retired) cudaFree(p);
        if (b->codes_done) cudaEventDestroy(b->codes_done);
        for (auto& e : b->legs) { cudaFree(e.buf); cudaEventDestroy(e.ready); }
    }
    delete b;
    return SGMM_OK;
}

static int check_rollout_args(const sgmm_bundle* bundle, const sgmm_population* mm, const sgmm_population* adv,
                              const sgmm_rollout_params* params, const double* fitness, const int32_t* trades)
{
    if (!bundle || !mm || !params) { set_error("NULL bundle / mm / params"); return SGMM_ERR_INVALID; }
    if (mm->count > 0 && (!fitness || !trades)) { set_error("NULL output array"); return SGMM_ERR_INVALID; }
    if (params->precision != SGMM_PRECISION_F32 && params->precision != SGMM_PRECISION_BF16 && params->precision != SGMM_PRECISION_TF32 && params->precision != SGMM_PRECISION_F16 && params->precision != SGMM_PRECISION_EXACT) { set_error("unknown precision %d", params->precision); return SGMM_ERR_INVALID; }
    if (mm->hidden == 256) {
        if (params->precision != SGMM_PRECISION_BF16 && params->precision != SGMM_PRECISION_EXACT) { set_error("hidden=256: pass precision=SGMM_PRECISION_EXACT (bit-exact SGMM-F32 order) or SGMM_PRECISION_BF16 (tensor cores); F32 and TF32 are H=32 paths"); return SGMM_ERR_UNSUPPORTED; }
    } else if (mm->hidden == 32) {
    } else if (params->precision != SGMM_PRECISION_F32) { set_error("precision %d needs hidden=32 or hidden=256 (EXACT, BF16) or hidden=32 (TF32, F16)", params->precision); return SGMM_ERR_UNSUPPORTED; }
    if (adv && adv->count != mm->count) { set_error("adv.count (%lld) != mm.count (%lld): MM i meets adversary i (Env/drl_engine.py:115)", (long long)adv->count, (long long)mm->count); return SGMM_ERR_INVALID; }
    if (adv && adv->hidden != 32) { set_error("adversary genomes are 1250-float TradingPolicy(32) genomes (models/model.py:63)"); return SGMM_ERR_INVALID; }
    return SGMM_OK;
}

int sgmm_rollout_population(const sgmm_bundle* bundle, const sgmm_population* mm, const sgmm_population* adv,
                            const sgmm_rollout_params* params, double* fitness, int32_t* trades, void* stream)
{
    if (int rc = check_rollout_args(bundle, mm, adv, params, fitness, trades)) return rc;
    PopArgs pm, pa;
    if (int rc = fill_pop(mm, "mm", pm)) return rc;
    if (adv) if (int rc = fill_pop(adv, "adv", pa)) return rc;
    DeviceGuard guard(bundle->device);
    return launch_population(bundle, pm, adv ? &pa : nullptr, mm->hidden, params->precision, params->phi, params->fee_rate,
                             params->units_per_lane, params->warps_per_cta, fitness, trades, (cudaStream_t)stream);
}

int sgmm_rollout_tc_audit(const sgmm_bundle* bundle, const sgmm_population* mm, const sgmm_population* adv,
                          const sgmm_rollout_params* params, double* fitness, int32_t* trades, float* raw_table,
                          int32_t* act_trace, void* stream)
{
    if (int rc = check_rollout_args(bundle, mm, adv, params, fitness, trades)) return rc;
    if (params->precision == SGMM_PRECISION_F32 || params->precision == SGMM_PRECISION_EXACT) { set_error("audit entry is for the tensor-core paths (precision BF16 / TF32 / F16)"); return SGMM_ERR_INVALID; }
    PopArgs pm, pa;
    if (int rc = fill_pop(mm, "mm", pm)) return rc;
    if (adv) if (int rc = fill_pop(adv, "adv", pa)) return rc;
    DeviceGuard guard(bundle->device);
    if (mm->hidden == 32)
        return launch_tc32(bundle, pm, adv ? &pa : nullptr, params->phi, params->fee_rate, params->units_per_lane, fitness, trades, raw_table,
                           act_trace, (cudaStream_t)stream, tc32_mode_of(params->precision));
    if (adv)
        return launch_spec256_adv(bundle, pm, pa, params->phi, params->fee_rate, fitness, trades, raw_table, act_trace, (cudaStream_t)stream);
    return launch_spec256(bundle, pm, params->phi, params->fee_rate, fitness, trades, raw_table, act_trace, (cudaStream_t)stream);
}

int sgmm_rollout_spec256_audit(const sgmm_bundle* bundle, const sgmm_population* mm, const sgmm_rollout_params* params,
                               double* fitness, int32_t* trades, float* raw_table, int32_t* act_trace, void* stream)
{
    return sgmm_rollout_tc_audit(bundle, mm, nullptr, params, fitness, trades, raw_table, act_trace, stream);
}

// One host-buffer rollout enqueued on `st` using workspace slot `slot` of the bundle: H2D genomes, kernel(s), D2H results.
// No synchronisation; the caller holds the slot's mutex-free ownership (the public entries serialise per slot).
static int enqueue_host_rollout(sgmm_bundle* b, int slot, const sgmm_population* mm, const sgmm_population* adv,
                                const sgmm_rollout_params* params, double* fitness, int32_t* trades, cudaStream_t st)
{
    const int64_t P = mm->count, G = genome_len(mm->hidden), GA = 1250;
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t mm_bytes = align((size_t)(mm->genomes ? P * G : G) * sizeof(float));
    const size_t adv_bytes = adv ? align((size_t)(adv->genomes ? P * GA : GA) * sizeof(float)) : 0;
    const size_t fit_bytes = align((size_t)P * sizeof(double)), trd_bytes = align((size_t)P * sizeof(int32_t));
    if (int rc = ensure_workspace(b, slot, mm_bytes + adv_bytes + fit_bytes + trd_bytes)) return rc;
    char* base = (char*)b->ws[slot];
    float* d_mm = (float*)base; float* d_adv = (float*)(base + mm_bytes);
    double* d_fit = (double*)(base + mm_bytes + adv_bytes); int32_t* d_trd = (int32_t*)(base + mm_bytes + adv_bytes + fit_bytes);
    PopArgs pm, pa;
    if (int rc = fill_pop(mm, "mm", pm)) return rc;
    const float* hsrc = mm->genomes ? mm->genomes : mm->master;
    if (int rc = check_cuda(cudaMemcpyAsync(d_mm, hsrc, (size_t)(mm->genomes ? P * G : G) * sizeof(float), cudaMemcpyHostToDevice, st), "H2D genomes")) return rc;
    if (mm->genomes) pm.genomes = d_mm; else pm.master = d_mm;
    if (adv) {
        if (int rc = fill_pop(adv, "adv", pa)) return rc;
        const float* asrc = adv->genomes ? adv->genomes : adv->master;
        if (int rc = check_cuda(cudaMemcpyAsync(d_adv, asrc, (size_t)(adv->genomes ? P * GA : GA) * sizeof(float), cudaMemcpyHostToDevice, st), "H2D adversary genomes")) return rc;
        if (adv->genomes) pa.genomes = d_adv; else pa.master = d_adv;
    }
    if (int rc = launch_population(b, pm, adv ? &pa : nullptr, mm->hidden, params->precision, params->phi, params->fee_rate,
                                   params->units_per_lane, params->warps_per_cta, d_fit, d_trd, st)) return rc;
    if (int rc = check_cuda(cudaMemcpyAsync(fitness, d_fit, (size_t)P * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H fitness")) return rc;
    return check_cuda(cudaMemcpyAsync(trades, d_trd, (size_t)P * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "D2H trades");
}

int sgmm_rollout_population_host(const sgmm_bundle* bundle, const sgmm_population* mm, const sgmm_population* adv,
                                 const sgmm_rollout_params* params, double* fitness, int32_t* trades, void* stream)
{
    if (int rc = check_rollout_args(bundle, mm, adv, params, fitness, trades)) return rc;
    if (mm->count == 0) return SGMM_OK;
    sgmm_bundle* b = const_cast<sgmm_bundle*>(bundle);
    std::lock_guard<std::mutex> lock(b->ws_mutex);
    DeviceGuard guard(b->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = enqueue_host_rollout(b, 0, mm, adv, params, fitness, trades, st)) return rc;
    return check_cuda(cudaStreamSynchronize(st), "rollout_population_host");
}

int sgmm_rollout_population_host_async(const sgmm_bundle* bundle, const sgmm_population* mm, const sgmm_population* adv,
                                       const sgmm_rollout_params* params, double* fitness, int32_t* trades, int32_t* ticket)
{
    if (!ticket) { set_error("ticket is NULL"); return SGMM_ERR_INVALID; }
    *ticket = -1;
    if (int rc = check_rollout_args(bundle, mm, adv, params, fitness, trades)) return rc;
    sgmm_bundle* b = const_cast<sgmm_bundle*>(bundle);
    std::lock_guard<std::mutex> lock(b->ws_mutex);
    DeviceGuard guard(b->device);
    // slots 1 .. SGMM_HOST_SLOTS-1 rotate; a slot is reused only after its previous batch has completed
    const int slot = 1 + (int)(b->async_next++ % (SGMM_HOST_SLOTS - 1));
    if (!b->slot_stream[slot])
        if (int rc = check_cuda(cudaStreamCreateWithFlags(&b->slot_stream[slot], cudaStreamNonBlocking), "cudaStreamCreate(slot)")) return rc;
    cudaStream_t st = b->slot_stream[slot];
    if (int rc = check_cuda(cudaStreamSynchronize(st), "slot still busy")) return rc;       // its previous batch (if any) is done
    if (mm->count > 0)
        if (int rc = enqueue_host_rollout(b, slot, mm, adv, params, fitness, trades, st)) return rc;
    *ticket = slot;
    return SGMM_OK;
}

int sgmm_rollout_wait(const sgmm_bundle* bundle, int32_t ticket)
{
    if (!bundle || ticket < 1 || ticket >= SGMM_HOST_SLOTS) { set_error("bad bundle / ticket"); return SGMM_ERR_INVALID; }
    sgmm_bundle* b = const_cast<sgmm_bundle*>(bundle);
    cudaStream_t st;
    { std::lock_guard<std::mutex> lock(b->ws_mutex); st = b->slot_stream[ticket]; }
    if (!st) { set_error("ticket %d was never issued", ticket); return SGMM_ERR_INVALID; }
    DeviceGuard guard(b->device);
    return check_cuda(cudaStreamSynchronize(st), "rollout_wait");
}

int sgmm_rollout_trace(const sgmm_bundle* bundle, const float* mm_genome, int32_t hidden, const float* adv_genome,
                       const int32_t* forced_actions, const sgmm_rollout_params* params, const sgmm_trace* trace,
                       double* fitness, int32_t* trades, void* stream)
{
    if (!bundle || !params) { set_error("NULL bundle / params"); return SGMM_ERR_INVALID; }
    DeviceGuard guard(bundle->device);
    return launch_trace(bundle, mm_genome, hidden, adv_genome, forced_actions, nullptr, params->phi, params->fee_rate,
                        trace, fitness, trades, (cudaStream_t)stream);
}

int sgmm_rollout_trace_population(const sgmm_bundle* bundle, const sgmm_population* mm, const sgmm_population* adv,
                                  const sgmm_rollout_params* params, const sgmm_trace* trace, double* fitness, int32_t* trades,
                                  void* stream)
{
    if (!params) { set_error("NULL bundle / mm / params"); return SGMM_ERR_INVALID; }
    if (params->precision == SGMM_PRECISION_BF16 || params->precision == SGMM_PRECISION_TF32 || params->precision == SGMM_PRECISION_F16) {
        set_error("the population trace runs in SGMM-F32 order: pass precision SGMM_PRECISION_F32 or SGMM_PRECISION_EXACT (tensor-core traces are not built)");
        return SGMM_ERR_UNSUPPORTED;
    }
    sgmm_rollout_params exact = *params;                    // F32 and EXACT are the same trace at either width
    if (exact.precision == SGMM_PRECISION_F32) exact.precision = SGMM_PRECISION_EXACT;
    if (int rc = check_rollout_args(bundle, mm, adv, &exact, fitness, trades)) return rc;
    if (mm->count == 0) return SGMM_OK;
    PopArgs pm, pa;
    if (int rc = fill_pop(mm, "mm", pm)) return rc;
    if (adv) if (int rc = fill_pop(adv, "adv", pa)) return rc;
    DeviceGuard guard(bundle->device);
    return launch_trace_population(bundle, pm, adv ? &pa : nullptr, mm->hidden, params->phi, params->fee_rate, trace, fitness, trades,
                                   (cudaStream_t)stream);
}

int sgmm_rollout_table(const sgmm_bundle* bundle, const int32_t* table, const sgmm_rollout_params* params,
                       const sgmm_trace* trace, double* fitness, int32_t* trades, void* stream)
{
    if (!bundle || !params || !table) { set_error("NULL bundle / params / table"); return SGMM_ERR_INVALID; }
    DeviceGuard guard(bundle->device);
    return launch_trace(bundle, nullptr, 32, nullptr, nullptr, table, params->phi, params->fee_rate,
                        trace, fitness, trades, (cudaStream_t)stream);
}

int sgmm_bundle_windows(int64_t n_events, const double* askprice1, const double* bidprice1, const double* p_buy_max,
                        const double* p_sell_min, int64_t event_step, int64_t n_signals, double* mid_next, double* best_ask,
                        double* best_bid, double* buy_max, double* sell_min, void* stream)
{
    if (n_events > 0 && n_signals > 1 && (!askprice1 || !bidprice1 || !p_buy_max || !p_sell_min || !mid_next || !best_ask || !best_bid || !buy_max || !sell_min)) {
        set_error("NULL array"); return SGMM_ERR_INVALID;
    }
    return launch_bundle_windows(n_events, askprice1, bidprice1, p_buy_max, p_sell_min, event_step, n_signals,
                                 mid_next, best_ask, best_bid, buy_max, sell_min, (cudaStream_t)stream);
}

int sgmm_bundle_windows_host(int64_t n_events, const double* askprice1, const double* bidprice1, const double* p_buy_max,
                             const double* p_sell_min, int64_t event_step, int64_t n_signals, double* mid_next, double* best_ask,
                             double* best_bid, double* buy_max, double* sell_min, int device, void* stream)
{
    if (n_events < 0 || n_signals < 0 || event_step <= 0) { set_error("negative size / non-positive step"); return SGMM_ERR_INVALID; }
    if (n_signals <= 1 || n_events == 0) return SGMM_OK;
    if ((n_events + event_step - 1) / event_step < n_signals) { set_error("more signals than sampled events"); return SGMM_ERR_INVALID; }
    if (!askprice1 || !bidprice1 || !p_buy_max || !p_sell_min || !mid_next || !best_ask || !best_bid || !buy_max || !sell_min) { set_error("NULL array"); return SGMM_ERR_INVALID; }
    DeviceGuard guard(device);
    if (!guard.ok) { set_error("cannot select CUDA device %d", device); return SGMM_ERR_CUDA; }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t e = (size_t)n_events, nb = (size_t)(n_signals - 1);
    double* d = nullptr;
    int rc = check_cuda(cudaMalloc(&d, (4 * e + 5 * nb) * sizeof(double)), "cudaMalloc(windows)");
    const double* src[4] = {askprice1, bidprice1, p_buy_max, p_sell_min};
    for (int k = 0; k < 4 && !rc; ++k) rc = check_cuda(cudaMemcpyAsync(d + k * e, src[k], e * sizeof(double), cudaMemcpyHostToDevice, st), "H2D events");
    double* o = d + 4 * e;
    if (!rc) rc = launch_bundle_windows(n_events, d, d + e, d + 2 * e, d + 3 * e, event_step, n_signals, o, o + nb, o + 2 * nb, o + 3 * nb, o + 4 * nb, st);
    double* dst[5] = {mid_next, best_ask, best_bid, buy_max, sell_min};
    for (int k = 0; k < 5 && !rc; ++k) rc = check_cuda(cudaMemcpyAsync(dst[k], o + k * nb, nb * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H bars");
    if (!rc) rc = check_cuda(cudaStreamSynchronize(st), "bundle_windows_host");
    cudaFree(d);
    return rc;
}

int sgmm_trace_analytics(int64_t n_traces, int64_t n_steps, const double* wealth, const double* cash, const double* mid,
                         const int32_t* inventory, const uint8_t* is_trade, double* scratch, double* out, void* stream)
{
    return launch_analytics(n_traces, n_steps, wealth, cash, mid, inventory, is_trade, scratch, out, (cudaStream_t)stream);
}

int sgmm_trace_analytics_host(int64_t n_traces, int64_t n_steps, const double* wealth, const int32_t* inventory,
                              const uint8_t* is_trade, double* out, int device, void* stream)
{
    if (n_traces < 0 || n_steps < 0) { set_error("negative size"); return SGMM_ERR_INVALID; }
    if (n_traces == 0) return SGMM_OK;
    if (!out || (n_steps > 0 && (!wealth || !inventory || !is_trade))) { set_error("NULL array"); return SGMM_ERR_INVALID; }
    DeviceGuard guard(device);
    if (!guard.ok) { set_error("cannot select CUDA device %d", device); return SGMM_ERR_CUDA; }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)n_traces * (size_t)n_steps;
    char* d = nullptr;
    const size_t bytes = 2 * n * sizeof(double) + n * sizeof(int32_t) + ((n + 7) & ~(size_t)7) + (size_t)n_traces * 6 * sizeof(double) + 64;
    int rc = check_cuda(cudaMalloc(&d, bytes), "cudaMalloc(analytics)");
    double* dw = (double*)d; double* ds = dw + n; double* dout = ds + n;
    int32_t* di = (int32_t*)(dout + (size_t)n_traces * 6); uint8_t* dt = (uint8_t*)(di + n);
    if (!rc && n) rc = check_cuda(cudaMemcpyAsync(dw, wealth, n * sizeof(double), cudaMemcpyHostToDevice, st), "H2D wealth");
    if (!rc && n) rc = check_cuda(cudaMemcpyAsync(di, inventory, n * sizeof(int32_t), cudaMemcpyHostToDevice, st), "H2D inventory");
    if (!rc && n) rc = check_cuda(cudaMemcpyAsync(dt, is_trade, n, cudaMemcpyHostToDevice, st), "H2D is_trade");
    if (!rc) rc = launch_analytics(n_traces, n_steps, dw, nullptr, nullptr, di, dt, ds, dout, st);
    if (!rc) rc = check_cuda(cudaMemcpyAsync(out, dout, (size_t)n_traces * 6 * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H summary");
    if (!rc) rc = check_cuda(cudaStreamSynchronize(st), "trace_analytics_host");
    cudaFree(d);
    return rc;
}

int sgmm_env_init(sgmm_env_state* e, double phi, double tick_size, double fee_rate)
{
    if (!e) { set_error("env is NULL"); return SGMM_ERR_INVALID; }
    e->fee_rate = fee_rate; e->phi = phi; e->tick_size = tick_size;     // market_env.py:9-11
    e->inventory = 0; e->cash = 0.0; e->i_max = 2; e->i_min = -2;       // :12-15
    return SGMM_OK;
}

int sgmm_env_step_host(sgmm_env_state* e, const int64_t action[2], const int64_t* adv_action, double mid_next,
                       double best_ask, double best_bid, double buy_max, double sell_min, sgmm_step_info* info)
{
    if (!e || !action || !info) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    int64_t off_a = action[0], off_b = action[1];                        // market_env.py:23
    if (adv_action) { off_a += adv_action[0]; off_b += adv_action[1]; }  // :25-28
    env_step<int64_t>(*e, off_a, off_b, mid_next, best_ask, best_bid, buy_max, sell_min, *info);
    return SGMM_OK;
}

int sgmm_env_step_host_real(sgmm_env_state* e, const double action[2], const int64_t* adv_action, double mid_next,
                            double best_ask, double best_bid, double buy_max, double sell_min, sgmm_step_info* info)
{
    if (!e || !action || !info) { set_error("NULL argument"); return SGMM_ERR_INVALID; }
    double off_a = action[0], off_b = action[1];                         // market_env.py:23 (offsets as given)
    if (adv_action) { off_a = add_rn(off_a, (double)adv_action[0]); off_b = add_rn(off_b, (double)adv_action[1]); }  // :25-28
    env_step<double>(*e, off_a, off_b, mid_next, best_ask, best_bid, buy_max, sell_min, *info);
    return SGMM_OK;
}

}  // extern "C"
