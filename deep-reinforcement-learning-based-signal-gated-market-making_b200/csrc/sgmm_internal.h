// sgmm_internal.h -- shared declarations between the translation units of libsgmm_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <mutex>
#include <vector>
#include "../../include/sgmm.h"

namespace sgmm {

// One bar as the kernels see it.  16 B signal/threshold record + 32 B price record.
struct __align__(32) BarSig {
    float z1, z2;        // normalised SGU1 / SGU2 signals (drl_engine.py:33-34), fp32
    float tha, thb;      // float fill thresholds on q = raw*5 (BEFORE rounding):
                         //   fill_sell <=> q_a < tha, fill_buy <=> q_b < thb   (-inf never, +inf always)
                         // tha = Ka + 0.5 nudged one ulp up when Ka is even (|Ka| >= 2^23: the float
                         // after the largest float <= Ka), so that the strict compare reproduces
                         // round-half-even followed by off <= Ka
    int32_t ka1, kb1;    // integer thresholds + 1: fill_sell <=> off_a < ka1 (used when the adversary
    int32_t pad0, pad1;  // displaces the rounded offsets); INT32_MIN never, INT32_MAX always
};
struct __align__(32) BarPx {
    double ask, bid, mid_next, pad;
};

// step code of the deferred fp64 accounting (sgmm_account.cu): this value in an offset field = that side did not fill
#define SGMM_CODE_NOFILL INT32_MIN
#define SGMM_CODE_NOFILL_F ((int)0xFFFFFFFF)     // the same marker when the field carries the fp32 q = raw*5 (a NaN)
constexpr int32_t K_NEVER = INT32_MIN;
constexpr int32_t K_ALWAYS = INT32_MAX;
constexpr int32_t K_CLAMP = 1 << 30;

}  // namespace sgmm

#define SGMM_HOST_SLOTS 3          // 1 synchronous + 2 pipelined host-buffer workspaces per bundle

struct sgmm_bundle {
    int device = 0;
    int64_t T = 0;
    double tick = 0.0;
    sgmm::BarSig* sig = nullptr;       // [T]
    sgmm::BarPx* px = nullptr;         // [T]
    double* bmax = nullptr;            // [T] raw bounds (trace kernel runs the literal step core)
    double* smin = nullptr;
    uint8_t* a1 = nullptr;             // [ceil(T/25)][4096] layer-1 A operand tiles of the tensor-core H=32 path (sgmm_tc32.cu)
    // grow-only workspaces of the *_host entry points: slot 0 = the synchronous entry (caller's stream), slots 1.. = the
    // pipelined entry (sgmm_rollout_population_host_async), each with its own stream so that the H2D copy of one batch
    // overlaps the kernel of the previous one
    std::mutex ws_mutex;
    void* ws[SGMM_HOST_SLOTS] = {};
    size_t ws_bytes[SGMM_HOST_SLOTS] = {};
    cudaStream_t slot_stream[SGMM_HOST_SLOTS] = {};
    uint64_t async_next = 0;
    // [count][T] 64-bit step codes of the tensor-core rollouts (sgmm_account.cu), grow-only
    std::mutex codes_mutex;
    uint64_t* codes = nullptr;
    size_t codes_cap = 0;
    std::vector<uint64_t*> codes_retired;
    // leg tables of the tensor-core H=32 rollout (sgmm_tc32.cu): one per fee rate seen, never freed before the bundle
    struct LegTable { double fee; void* buf; cudaEvent_t ready; cudaStream_t stream; };
    std::mutex legs_mutex;
    std::vector<LegTable> legs;
    // ordering of the users of `codes` across streams: the last user's stream and an event recorded after its accounting
    // kernel; a rollout arriving on another stream waits for it (outside stream capture)
    cudaStream_t codes_stream = nullptr;
    cudaEvent_t codes_done = nullptr;
    bool codes_busy = false;
    bool codes_captured = false;       // a stream capture has used `codes`: its address may live in a graph
};

namespace sgmm {

// device-side population descriptor
struct PopArgs {
    const float* genomes;   // [count,G] or nullptr
    const float* master;    // [G]
    const int64_t* first_index_dev;   // optional device scalar added to first_index (GA: best child)
    float sigma;
    const float* sigma_dev;           // optional device scalar overriding sigma (GA sigma decay)
    uint64_t seed;
    uint64_t generation;
    const int32_t* generation_dev;    // optional device scalar overriding generation
    int64_t first_index;
    int64_t count;
};

struct RolloutArgs {
    const BarSig* sig;
    const BarPx* px;
    int64_t T;
    double tick, phi, fee;
    PopArgs mm, adv;
    double* fitness;
    int32_t* trades;
    uint64_t* codes;     // [count][T] step codes (sgmm_account.cu)
};

void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

inline int64_t genome_len(int H) { return (int64_t)H * H + 7 * (int64_t)H + 2; }

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute of a kernel: opt in once per (kernel, device).
// `mask` is one static word per kernel instantiation, bit d = configured on device d (the calling thread's current
// device).  Devices >= 64 simply re-apply the attribute on every launch.  Safe from concurrent host threads: a lost
// race only repeats an idempotent call.
template <typename Kernel>
inline int opt_in_smem(Kernel kern, size_t bytes, std::atomic<uint64_t>& mask, const char* what)
{
    int dev = -1;
    if (int rc = check_cuda(cudaGetDevice(&dev), "cudaGetDevice")) return rc;
    const bool tracked = dev >= 0 && dev < 64;
    if (tracked && (mask.load(std::memory_order_acquire) >> dev & 1ull)) return SGMM_OK;
    if (int rc = check_cuda(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes), what)) return rc;
    if (tracked) mask.fetch_or(1ull << dev, std::memory_order_release);
    return SGMM_OK;
}

int launch_rollout(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, int hidden,
                   double phi, double fee, int units_per_lane, int warps_per_cta,
                   double* fitness, int32_t* trades, cudaStream_t st);
// small populations, fast (sgmm_one.cu): policy table for every (bar, inventory) + automaton scan + reference-order sum
constexpr int64_t SMALL_POP_MAX = 400;      // measured break-even against the sequential kernel: ~420 individuals (profiles/r2_small_population_path.log)
constexpr int64_t SMALL_POP_MAX_ADV = 148;  // with the adversary (one 512-thread CTA per individual and SM)
int launch_rollout_small(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, double phi, double fee, double* fitness, int32_t* trades,
                         cudaStream_t st);
// the policy table of the small-population path for mm.count individuals (sgmm_one.cu), in the format of `mode`: 0 step code
// + next inventory, 1 q = raw*5 per (bar, inventory) (adversary walk), 2 raw outputs per (bar, inventory) (population trace)
int launch_policy_table(const sgmm_bundle* b, const PopArgs& mm, int mode, float2* code, uint8_t* next, cudaStream_t st);
// the walk + fp64 half of the policy-table path over tables code [P][T][5] / next [P][T][8] (sgmm_one.cu)
int launch_walk(const sgmm_bundle* b, int64_t P, const float2* code, const uint8_t* next, const PopArgs* adv, double phi, double fee,
                double* fitness, int32_t* trades, cudaStream_t st);
// the market maker's offsets before the adversary's displacement along the Walk20 walk of q tables [P][T][5] (audit, sgmm_one.cu)
int launch_adv_offsets(const sgmm_bundle* b, int64_t P, const float2* code, const PopArgs& adv, int32_t* act_trace, cudaStream_t st);
// H = 256 populations as batches of policy table + walk (sgmm_exact256.cu, and sgmm_spec256.cu with the adversary).  The
// scratch of a batch, `per_ind` 8-byte words per individual, is the bundle's code buffer (ordered rollouts per bundle; the
// first rollout of a size must not run under a stream capture) and stays under the byte budget SGMM_EXACT256_BATCH_BYTES
// (environment, read on every call; default 2 GiB): *nb individuals per batch.
int reserve_batches(const sgmm_bundle* b, int64_t P, int64_t per_ind, cudaStream_t st, int64_t* nb, uint64_t** buf);
// Batches of at most nb individuals of genome length G: fn(pm, pa, b0) gets individuals b0 .. b0+n-1 of mm / adv as pm / pa
// (pa nullptr without the adversary).
template <class Fn>
int for_each_batch(const PopArgs& mm, const PopArgs* adv, int64_t nb, int64_t G, Fn fn)
{
    for (int64_t b0 = 0; b0 < mm.count; b0 += nb) {
        const int64_t n = mm.count - b0 < nb ? mm.count - b0 : nb;
        PopArgs pm = mm;
        if (pm.genomes) pm.genomes += b0 * G; else pm.first_index += b0;
        pm.count = n;
        PopArgs pa{};
        if (adv) {
            pa = *adv;
            if (pa.genomes) pa.genomes += b0 * 1250; else pa.first_index += b0;
            pa.count = n;
        }
        if (int rc = fn(pm, adv ? &pa : nullptr, b0)) return rc;
    }
    return SGMM_OK;
}
// Batches of at most nb individuals: table(pm, pa, b0) enqueues the policy table (code / next) of individuals b0 .. b0+n-1,
// pm / pa being those individuals of mm / adv (pa nullptr without the adversary); the walk then writes their fitness / trades.
template <class Table>
int walk_batches(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, int64_t nb, const float2* code, const uint8_t* next,
                 double phi, double fee, double* fitness, int32_t* trades, cudaStream_t st, Table table)
{
    return for_each_batch(mm, adv, nb, genome_len(256), [&](const PopArgs& pm, const PopArgs* pa, int64_t b0) {
        if (int rc = table(pm, pa, b0)) return rc;
        return launch_walk(b, pm.count, code, next, pa, phi, fee, fitness + b0, trades + b0, st);
    });
}
// bit-exact H = 256 (sgmm_exact256.cu): batches of policy table + walk; and the raw-output table of one genome for the trace
int launch_exact256(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, double phi, double fee, double* fitness, int32_t* trades,
                    cudaStream_t st);
namespace x256 {
// the exact H = 256 policy table of `count` 8-byte aligned genome rows (modes as launch_policy_table), and the staging of
// seeded children or unaligned rows into such rows (sgmm_exact256.cu)
int launch_table(const sgmm_bundle* b, const float* rows, int64_t count, int mode, float2* code, uint8_t* next, cudaStream_t st);
int launch_stage(const sgmm_bundle* b, const PopArgs& mm, int64_t count, float* out, cudaStream_t st);
bool needs_stage(const PopArgs& mm);
}
int launch_exact256_raw(const sgmm_bundle* b, const float* genome, float2* out, float* stage_buf, cudaStream_t st);
int launch_trace(const sgmm_bundle* b, const float* mm_genome, int hidden, const float* adv_genome,
                 const int32_t* forced, const int32_t* table, double phi, double fee, const sgmm_trace* tr,
                 double* fitness, int32_t* trades, cudaStream_t st);
// recorder traces of a population, H = 32 or 256 in SGMM-F32 order, [count][T] per column (sgmm_trace_pop.cu)
int launch_trace_population(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, int hidden, double phi, double fee,
                            const sgmm_trace* tr, double* fitness, int32_t* trades, cudaStream_t st);
int launch_spec256(const sgmm_bundle* b, const PopArgs& mm, double phi, double fee, double* fitness, int32_t* trades,
                   float* raw_table, int32_t* act_trace, cudaStream_t st);
// H = 256 on the tensor cores with the adversary: spec256 q tables walked by walk_account_kernel<Walk20>, in batches
int launch_spec256_adv(const sgmm_bundle* b, const PopArgs& mm, const PopArgs& adv, double phi, double fee, double* fitness,
                       int32_t* trades, float* raw_table, int32_t* act_trace, cudaStream_t st);
int launch_tc32(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, double phi, double fee, int group, double* fitness, int32_t* trades,
                float* raw_table, int32_t* act_trace, cudaStream_t st, int mode = 0);   // mode: 0 bf16, 1 tf32, 2 f16
// the rollout of a population on the kernel that serves (hidden, precision, adversary) (sgmm_capi.cu); units_per_lane is
// the tensor-core group size at H = 32 in BF16 / TF32 / F16.  The arguments are checked by the caller.
int launch_population(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, int hidden, int precision, double phi, double fee,
                      int units_per_lane, int warps_per_cta, double* fitness, int32_t* trades, cudaStream_t st);
int launch_tc32_prologue(sgmm_bundle* b, cudaStream_t st);
int launch_account(const sgmm_bundle* b, const uint64_t* codes, int64_t count, double phi, double fee, double* fitness,
                   int32_t* trades, cudaStream_t st, bool float_offsets = false);
int reserve_codes(const sgmm_bundle* b, int64_t count, cudaStream_t st, uint64_t** out);
int release_codes(const sgmm_bundle* b, cudaStream_t st);      // after the last kernel that reads the codes was enqueued
// Scope guard of a successful reserve_codes / reserve_batches: done() is release_codes on the success path; any other exit
// (an error return after some kernels were enqueued) still records the bundle's event on `st`, so that the next user on
// another stream waits for the work already enqueued.  The error message of that exit is kept.
struct CodesRelease {
    const sgmm_bundle* b;
    cudaStream_t st;
    bool pending = true;
    CodesRelease(const sgmm_bundle* bundle, cudaStream_t stream) : b(bundle), st(stream) {}
    CodesRelease(const CodesRelease&) = delete;
    CodesRelease& operator=(const CodesRelease&) = delete;
    int done() { pending = false; return release_codes(b, st); }
    ~CodesRelease();
};
size_t tc32_a1_bytes(int64_t T);
int launch_prologue(sgmm_bundle* b, const float* z1, const float* z2, const double* mid,
                    const double* ask, const double* bid, cudaStream_t st);

int launch_bundle_windows(int64_t E, const double* ask1, const double* bid1, const double* pmax, const double* pmin,
                          int64_t step, int64_t n, double* mid_next, double* best_ask, double* best_bid,
                          double* buy_max, double* sell_min, cudaStream_t st);
int launch_analytics(int64_t B, int64_t T, const double* wealth, const double* cash, const double* mid,
                     const int32_t* inventory, const uint8_t* is_trade, double* scratch, double* out, cudaStream_t st);

}  // namespace sgmm
