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
    // grow-only scratch of one call at a time: [count][T] 64-bit step codes, policy tables (ScratchLease, sgmm_account.cu)
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

// Device state of one GA run (sgmm_ga.cu); a sweep of K runs keeps K of them, contiguous.  seed / patience / phi / fee are
// set at creation and read by the sweep's table and walk kernels (sgmm_one.cu) and by ga_tell_kernel / ga_update_kernel.
struct GaDev {
    int32_t generation;
    int32_t stale;
    float sigma, adv_sigma;
    double best_val;
    int64_t best_idx, adv_best_idx;
    double train_f; int32_t train_trades; int32_t patience;
    uint64_t seed;
    double phi, fee;             // the walk reads the fee as stored: -0.0 and 0.0 stay distinct
};

constexpr uint64_t ADV_SEED_FLIP = 0x8000000000000000ull;   // adversary noise stream (same as the oracle)

// The seeded children of a GA sweep (K runs of lambda children each, one launch): individual i of a launch is g = first + i
// of the sweep, child g % lambda of run r = g / lambda, regenerated from row r of `master` with run r's device sigma
// (adv_sigma when `adv`), generation and seed (seed ^ ADV_SEED_FLIP when `adv`) -- the child a solo GA of that run draws.
// The sweep's walks read run r's phi and fee from st[r].  With lambda = 1 and master = nullptr it only indexes the runs
// (validation of the K masters).
struct SweepPop {
    const float* master;       // [K][G] (G = 1250: the market makers' or the adversaries' masters)
    const GaDev* st;           // [K]
    int64_t lambda, first, count;
    int adv;
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

// Makes `dev` the calling thread's current device for the scope and restores the previous one; ok = the switch worked
struct DeviceGuard {
    int prev = -1; bool ok = false;
    explicit DeviceGuard(int dev) { if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess) ok = true; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// The SM count of `device`, queried once per device (sgmm_capi.cu).  A failed query is not cached and answers 148 (a B200);
// its error stays the thread's last CUDA error, so the launch check that follows reports it.
int sm_count(int device);

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
// objective: SGMM_OBJECTIVE_* (sgmm.h); a non-REWARD objective takes this route at every population size
int launch_rollout_small(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, double phi, double fee, double* fitness, int32_t* trades,
                         cudaStream_t st, int objective = SGMM_OBJECTIVE_REWARD);
// the policy table of the small-population path for mm.count individuals (sgmm_one.cu), in the format of `mode`: 0 step code
// + next inventory, 1 q = raw*5 per (bar, inventory) (adversary walk), 2 raw outputs per (bar, inventory) (population trace,
// PopArgs only).  Pop: PopArgs, or SweepPop (the children of a GA sweep).
template <class Pop>
int launch_policy_table(const sgmm_bundle* b, const Pop& mm, int mode, float2* code, uint8_t* next, cudaStream_t st);
// the walk + fp64 half of the policy-table path over tables code [P][T][5] / next [P][T][8] (sgmm_one.cu).  CTA i walks
// individual i of `pop`: with `adv` pop holds the adversaries (the 20-state walk over q tables; next unused); a SweepPop
// gives every CTA its run's phi and fee, a PopArgs takes phi / fee (and is not read without the adversary).  objective:
// SGMM_OBJECTIVE_* (sgmm.h); SHARPE needs obj_scratch [P][T] doubles, the others take nullptr.
template <class Pop>
int launch_walk(const sgmm_bundle* b, int64_t P, const float2* code, const uint8_t* next, const Pop& pop, bool adv, double phi,
                double fee, double* fitness, int32_t* trades, int objective, double* obj_scratch, cudaStream_t st);
// the market maker's offsets before the adversary's displacement along the Walk20 walk of q tables [P][T][5] (audit, sgmm_one.cu)
int launch_adv_offsets(const sgmm_bundle* b, int64_t P, const float2* code, const PopArgs& adv, int32_t* act_trace, cudaStream_t st);

// Scratch of one call in the bundle's grow-only code buffer (sgmm_account.cu).  Calls on one bundle take turns: an eager call
// on another stream than the buffer's last user waits for that user's event; under a stream capture the buffer cannot grow
// (the call is refused), and once a capture has used it an outgrown buffer is retired instead of freed.  Build the lease on
// (bundle, stream), reserve once, enqueue the kernels that use the scratch, then return done(): it records the event and
// reports its errors.  Any other exit after a successful reserve records the event in the destructor and keeps the error
// message of that exit.
class ScratchLease {
public:
    ScratchLease(const sgmm_bundle* b, cudaStream_t st) : b_(const_cast<sgmm_bundle*>(b)), st_(st) {}
    ScratchLease(const ScratchLease&) = delete;
    ScratchLease& operator=(const ScratchLease&) = delete;
    ~ScratchLease();
    // at least `words` 8-byte words at *out
    int reserve(int64_t words, uint64_t** out);
    // P individuals of per_ind words each, in batches under the byte budget SGMM_EXACT256_BATCH_BYTES (environment, read on
    // every call; default 2 GiB): *nb individuals per batch, nb * per_ind words at *out
    int reserve_in_batches(int64_t P, int64_t per_ind, int64_t* nb, uint64_t** out);
    int done();
private:
    sgmm_bundle* b_;
    cudaStream_t st_;
    bool pending_ = false;
};

// individuals b0 .. b0+n-1 of a population of genome length G
inline PopArgs batch_of(const PopArgs& p, int64_t b0, int64_t n, int64_t G)
{
    PopArgs r = p;
    if (r.genomes) r.genomes += b0 * G; else r.first_index += b0;
    r.count = n;
    return r;
}
inline SweepPop batch_of(const SweepPop& p, int64_t b0, int64_t n, int64_t)
{
    SweepPop r = p;
    r.first += b0;                                  // a batch may start inside a run: the kernels split first + i into (run, child)
    r.count = n;
    return r;
}
// Batches of at most nb individuals of genome length G: fn(pm, pa, b0) gets individuals b0 .. b0+n-1 of mm / adv as pm / pa
// (pa nullptr without the adversary).  Pop: PopArgs, or SweepPop (the children of a GA sweep).
template <class Pop, class Fn>
int for_each_batch(const Pop& mm, const Pop* adv, int64_t nb, int64_t G, Fn fn)
{
    for (int64_t b0 = 0; b0 < mm.count; b0 += nb) {
        const int64_t n = mm.count - b0 < nb ? mm.count - b0 : nb;
        const Pop pm = batch_of(mm, b0, n, G);
        Pop pa{};
        if (adv) pa = batch_of(*adv, b0, n, (int64_t)1250);
        if (int rc = fn(pm, adv ? &pa : nullptr, b0)) return rc;
    }
    return SGMM_OK;
}
// The scratch of one table-and-walk batch of n individuals: the policy table code [n][T][5], the next-inventory bytes
// [n][T][8] of the 5-state walk (nullptr when the table kind has none), then `extra` words per individual for the table
// callback (staged genomes), then the walk's objective scratch [n][T] (SGMM_OBJECTIVE_SHARPE only, else nullptr).
struct BatchScratch {
    float2* code;
    uint8_t* next;
    uint64_t* extra;
    double* obj;
};
// Episodes of mm.count individuals of genome length G as batches of policy table + walk in the bundle's code buffer
// (ScratchLease::reserve_in_batches).  table(pm, pa, b0, s) enqueues into s the table of individuals b0 .. b0+n-1, pm / pa being
// those individuals of mm / adv (pa nullptr without the adversary); the walk then writes their fitness / trades: over the
// adversaries pa, or else with individuals b0 .. b0+n-1 of `walk` as its CTAs' population -- mm itself, or the runs of a
// GA sweep whose phi and fee the CTAs take (launch_walk).  objective: what the walk writes as fitness (SGMM_OBJECTIVE_*);
// SHARPE adds T words per individual to the batch's scratch.
template <class Pop, class WalkPop, class Table>
int table_walk_batches(const sgmm_bundle* b, const Pop& mm, const Pop* adv, const WalkPop& walk, int64_t G, bool with_next,
                       int64_t extra, double phi, double fee, double* fitness, int32_t* trades, cudaStream_t st, Table table,
                       int objective = SGMM_OBJECTIVE_REWARD)
{
    if (mm.count == 0) return SGMM_OK;
    const int64_t T = b->T, table_words = (with_next ? 6 : 5) * T, obj_words = objective == SGMM_OBJECTIVE_SHARPE ? T : 0;
    ScratchLease lease(b, st);
    int64_t nb = 0;
    uint64_t* buf = nullptr;
    if (int rc = lease.reserve_in_batches(mm.count, table_words + extra + obj_words, &nb, &buf)) return rc;
    const BatchScratch s{reinterpret_cast<float2*>(buf), with_next ? reinterpret_cast<uint8_t*>(buf + nb * T * 5) : nullptr,
                         buf + nb * table_words, obj_words ? reinterpret_cast<double*>(buf + nb * (table_words + extra)) : nullptr};
    const int rc = for_each_batch(mm, adv, nb, G, [&](const Pop& pm, const Pop* pa, int64_t b0) {
        if (int rc = table(pm, pa, b0, s)) return rc;
        if (pa) return launch_walk(b, pm.count, s.code, nullptr, *pa, true, phi, fee, fitness + b0, trades + b0, objective, s.obj, st);
        return launch_walk(b, pm.count, s.code, s.next, batch_of(walk, b0, pm.count, G), false, phi, fee, fitness + b0,
                           trades + b0, objective, s.obj, st);
    });
    if (rc) return rc;
    return lease.done();
}
// GA sweeps at H = 32, exact (sgmm_one.cu).  launch_sweep_population: the mm.count seeded children of mm (and adv) on the
// policy-table path at every size, in batches (table_walk_batches); every walk CTA takes its run's phi and fee.
// launch_sweep_validation: K explicit masters [K][1250] (adversary off), walk CTA r with run r's phi and fee.
// objective: SGMM_OBJECTIVE_* of both (sgmm.h).
int launch_sweep_population(const sgmm_bundle* b, const SweepPop& mm, const SweepPop* adv, double* fitness, int32_t* trades,
                            cudaStream_t st, int objective);
int launch_sweep_validation(const sgmm_bundle* b, const float* masters, const GaDev* runs, int64_t K, double* fitness,
                            int32_t* trades, cudaStream_t st, int objective);
// bit-exact H = 256 (sgmm_exact256.cu): batches of policy table + walk; and the raw-output table of one genome for the trace
int launch_exact256(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, double phi, double fee, double* fitness, int32_t* trades,
                    cudaStream_t st, int objective = SGMM_OBJECTIVE_REWARD);
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
// the tensor-core group size at H = 32 in BF16 / TF32 / F16.  The arguments are checked by the caller.  A non-REWARD
// objective (SGMM_OBJECTIVE_*) takes the policy-table route (H = 32 F32 / EXACT, H = 256 EXACT); with a tensor-core
// precision it is SGMM_ERR_UNSUPPORTED.
int launch_population(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, int hidden, int precision, double phi, double fee,
                      int units_per_lane, int warps_per_cta, double* fitness, int32_t* trades, cudaStream_t st,
                      int objective = SGMM_OBJECTIVE_REWARD);
int launch_tc32_prologue(sgmm_bundle* b, cudaStream_t st);
int launch_account(const sgmm_bundle* b, const uint64_t* codes, int64_t count, double phi, double fee, double* fitness,
                   int32_t* trades, cudaStream_t st, bool float_offsets = false);
size_t tc32_a1_bytes(int64_t T);
int launch_prologue(sgmm_bundle* b, const float* z1, const float* z2, const double* mid,
                    const double* ask, const double* bid, cudaStream_t st);

int launch_bundle_windows(int64_t E, const double* ask1, const double* bid1, const double* pmax, const double* pmin,
                          int64_t step, int64_t n, double* mid_next, double* best_ask, double* best_bid,
                          double* buy_max, double* sell_min, cudaStream_t st);
int launch_analytics(int64_t B, int64_t T, const double* wealth, const double* cash, const double* mid,
                     const int32_t* inventory, const uint8_t* is_trade, double* scratch, double* out, cudaStream_t st);

}  // namespace sgmm
