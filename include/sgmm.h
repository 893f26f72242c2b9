/*
 * sgmm.h -- C ABI of the B200-native population rollout for signal-gated market making.
 *
 * The reference (KAS-W/Deep-Reinforcement-Learning-Based-Signal-Gated-Market-Making) has no FFI:
 * its boundary is a plain Python API.  Each entry point below names the reference interface it
 * replaces (paths relative to the reference root).  The Python package binds these with ctypes
 * (see INTEGRATION.md); no torch / C++ types cross this boundary.
 *
 * Conventions
 *   - every function returns SGMM_OK (0) or a negative SGMM_ERR_* code and never throws;
 *     sgmm_last_error() returns a thread-local human-readable message for the last failure.
 *   - "stream" is a cudaStream_t passed as void* (0 = legacy default stream).  Work is enqueued
 *     on it; functions taking DEVICE pointers never synchronise.  Functions taking HOST pointers
 *     (suffix _host, sgmm_bundle_create) copy through internal pinned staging buffers and
 *     synchronise the stream before returning.
 *   - the caller owns every buffer it passes in; the library owns only the opaque handles it
 *     creates (sgmm_*_create / sgmm_*_destroy).
 *   - genome layout = torch parameters() order of TradingPolicy(hidden=H) (models/model.py:28-36):
 *       W1[H,3] | b1[H] | W2[H,H] | b2[H] | W3[2,H] | b3[2]          G = H*H + 7H + 2 floats
 *     AdversaryPolicy (models/model.py:52-57) consumes the first 74 floats of a 1250-float genome:
 *       V1[12,3] | c1[12] | V2[2,12] | c2[2]
 *   - offsets: off_a widens the ask (ask + off_a*tick), off_b widens the bid (bid - off_b*tick)
 *     (Env/market_env.py:23,30-31).  Offsets are carried as int32 and clamped to +-2^30 ticks.
 */
#ifndef SGMM_H
#define SGMM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGMM_VERSION 101            /* 0.1.1 */

#define SGMM_OK               0
#define SGMM_ERR_INVALID     -1     /* bad argument (NULL, negative size, unsupported hidden width) */
#define SGMM_ERR_CUDA        -2     /* CUDA runtime failure; message carries cudaGetErrorString      */
#define SGMM_ERR_NOMEM       -3
#define SGMM_ERR_UNSUPPORTED -4     /* device is not sm_100 class / feature not built                */

/* precision of the policy MLP */
#define SGMM_PRECISION_F32   0      /* SGMM-F32 order on CUDA cores: bit-identical to the oracle (H=32) */
                                    /* The adversary (adv != NULL) runs on every H=32 path, tensor-core ones  */
                                    /* included (a 20-state automaton instead of a 5-state one), and at H=256 */
                                    /* with BF16 and EXACT.                                                    */
#define SGMM_PRECISION_BF16  1      /* policy layers on tcgen05 tensor cores, bf16 x bf16 -> fp32 in  */
                                    /* TMEM, all 5 inventories of every bar evaluated at once:        */
                                    /*   H=32  all three layers as GEMMs chained through TMEM         */
                                    /*         (sgmm_tc32.cu; params.units_per_lane = individuals per */
                                    /*         CTA group, even, 0 = auto)                             */
                                    /*   H=256 hidden and output layer (sgmm_spec256.cu: f16 operands,*/
                                    /*         f16 layer-2 accumulator, whatever tensor mode is asked)*/
                                    /*         With an adversary the kernel writes q = raw*5 of every */
                                    /*         (bar, inventory) and the 20-state walk of the exact    */
                                    /*         path runs over it, in batches of 40 B per individual   */
                                    /*         and bar under SGMM_EXACT256_BATCH_BYTES (see EXACT)    */
                                    /* policy outputs within a stated tolerance of the fp32 oracle;   */
                                    /* the env step given the offsets stays bit-exact                 */

#define SGMM_PRECISION_TF32  2      /* H=32 only: as BF16 but layers 2 and 3 on tcgen05 kind::tf32 (fp32  */
                                    /* activations in TMEM rounded to 10 mantissa bits, tf32 weights):    */
                                    /* ~4x tighter policy outputs at ~equal speed                        */

#define SGMM_PRECISION_F16   3      /* H=32 only: f16 operands AND f16 accumulators for layers 1-2 (read back  */
                                    /* packed, ReLU on f16 pairs, no conversion), fp32 for layer 3             */

#define SGMM_PRECISION_EXACT 4      /* SGMM-F32 order at every width the library builds (H=32 and H=256): bit-identical  */
                                    /* to the oracle, with or without the adversary.  H=32: the same route as F32.       */
                                    /* H=256: fp32 CUDA-core policy table of every (bar, inventory) + the automaton walk */
                                    /* (sgmm_exact256.cu), ~55x the time of the BF16 path.  Populations run in batches   */
                                    /* whose scratch (48 B per individual and bar, + 269 KB per seeded child) stays under */
                                    /* the byte budget SGMM_EXACT256_BATCH_BYTES (environment, read on every call;        */
                                    /* default 2 GiB).  F32 (0) with H=256 stays SGMM_ERR_UNSUPPORTED.                    */

/* rollout flags */
#define SGMM_FLAG_NONE       0

int sgmm_version(void);
const char* sgmm_last_error(void);
/* number of visible CUDA devices, or a negative error */
int sgmm_device_count(void);
int sgmm_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, uint64_t* total_mem);

/* ---------------------------------------------------------------------------------------------
 * Bundle: the device-resident bar set of one episode.
 * Replaces the 7-tuple returned by load_signals_bundle (pipeline/agent_trainer.py:75-77) as
 * consumed by evaluate_individual (Env/drl_engine.py:11).  z1/z2 are the NORMALISED signals
 * (Env/drl_engine.py:33-34) computed by the caller with its own numpy expression and cast to
 * float32; the other five arrays are float64, NaN allowed in buy_max / sell_min.
 * All pointers are HOST pointers of length T (T may be 0).  Besides uploading, creation runs the
 * prologue kernel that derives the integer fill thresholds
 *     Ka[t] = max{k : fl(ask + fl(k*tick)) <= buy_max}   Kb[t] = max{k : fl(bid - fl(k*tick)) >= sell_min}
 * with the reference's exact two-rounding fp64 expression (Env/market_env.py:30-31,37-38).
 * ------------------------------------------------------------------------------------------- */
typedef struct sgmm_bundle sgmm_bundle;

int sgmm_bundle_create(sgmm_bundle** out, int64_t T,
                       const float* z1, const float* z2, const double* mid_next,
                       const double* best_ask, const double* best_bid,
                       const double* buy_max, const double* sell_min,
                       double tick_size, int device, void* stream);
int sgmm_bundle_length(const sgmm_bundle* b, int64_t* T);
int sgmm_bundle_device(const sgmm_bundle* b, int* device);
/* copy the derived thresholds back (HOST int32[T] each, either may be NULL); INT32_MIN = never
 * fills, INT32_MAX = always fills */
int sgmm_bundle_thresholds(const sgmm_bundle* b, int32_t* ka, int32_t* kb, void* stream);
int sgmm_bundle_destroy(sgmm_bundle* b);

/* ---------------------------------------------------------------------------------------------
 * Population: who is evaluated.  Either explicit genomes [count, G] (the list returned by
 * NeuroEvolution.ask, models/model.py:65-71) or "children of a master": child i is
 *     master + sigma * N(0,1)[Philox4x32-10 key=seed, counter=(e/4, index_lo, index_hi, generation)]
 * generated inside the rollout kernel, index = first_index + i (so a sharded population draws
 * the same children whatever the number of ranks).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t hidden;          /* H; 32 for the reference policy (models/model.py:7)               */
    int32_t reserved;
    int64_t count;           /* P                                                                */
    const float* genomes;    /* [count, G] row-major, or NULL for seeded children                */
    const float* master;     /* [G], used when genomes == NULL                                   */
    float sigma;             /* mutation scale (models/model.py:61)                              */
    float reserved2;
    uint64_t seed;
    uint64_t generation;
    int64_t first_index;
} sgmm_population;

typedef struct {
    double phi;              /* inventory penalty (Env/market_env.py:10,57)                      */
    double fee_rate;         /* proportional fee  (Env/market_env.py:9,46,52)                    */
    int32_t precision;       /* SGMM_PRECISION_*                                                 */
    int32_t flags;           /* SGMM_FLAG_*                                                      */
    int32_t units_per_lane;  /* 0 = auto; 1, 2 or 4 hidden units per lane (tuning knob)          */
    int32_t warps_per_cta;   /* 0 = auto                                                         */
} sgmm_rollout_params;

/* Replaces Pool.starmap(evaluate_individual, zip(mm_pop, adv_pop)) (Env/drl_engine.py:104-115):
 * one full episode per individual, fitness[i] = total_reward (with the -50 no-trade penalty,
 * Env/drl_engine.py:64-65), trades[i] = number of steps with at least one fill (:60-61).
 * adv == NULL <=> use_arl False.  adv->count must equal mm->count (MM i meets adversary i).
 * All pointers inside mm / adv and fitness / trades are DEVICE pointers on the bundle's device.
 *
 * H = 256 rollouts are two kernels: the tensor-core rollout kernel does the policy and the integer half of the env step
 * and writes one 8-byte step code per bar into a grow-only scratch buffer OF THE BUNDLE ([count][T] codes); an
 * accounting kernel then does the reference's fp64 arithmetic (an FP64 instruction issued while tcgen05.mma executes
 * waits ~80x longer).  Consequences for the caller of H = 256 rollouts:
 *   - rollouts on one bundle share the scratch.  Eager calls on different streams are ordered by the library: a call on
 *     another stream than the last user of the buffer waits for that user's event.  Captured calls do not wait on
 *     events: the captures of one bundle must stay on one stream, and replays of a captured graph are ordered by the caller;
 *   - the first rollout of a given size allocates and therefore must not run under a stream capture (run one eagerly,
 *     then capture: under a capture a buffer too small is refused with SGMM_ERR_INVALID).  An outgrown buffer is freed
 *     (cudaFree, after every enqueued user) unless a capture has used the bundle's buffer: from then on outgrown buffers
 *     stay allocated until sgmm_bundle_destroy, so that a captured graph never holds a freed address.
 * H = 32 rollouts of more than 400 individuals are one kernel with no per-rollout scratch.  SMALL populations (up to 400
 * individuals, 148 with an adversary; exact precision, default launch geometry) take the policy-table path instead (the
 * exact policy for every (bar, inventory) in parallel + a prefix scan over the inventory automaton, bit-identical results):
 * its table ([count][T] x 48 B) lives in the same grow-only code buffer of the bundle, so the same two rules apply to them,
 * and to every SGMM_PRECISION_EXACT rollout at H = 256 (the same table path, in batches).
 * The tensor-core precisions with an adversary read a per-(bundle, fee_rate) table of the reference's exact fp64 P&L legs
 * (144 B per bar), built on the first such rollout: that first rollout must not run under a stream capture either (refused
 * with SGMM_ERR_INVALID).  Eager users on other streams wait for the build.  Fee rates are keyed by their bits (-0.0 and 0.0
 * are two tables); a bundle holds at most 64 of them, the 65th fee rate is SGMM_ERR_NOMEM. */
int sgmm_rollout_population(const sgmm_bundle* bundle, const sgmm_population* mm,
                            const sgmm_population* adv, const sgmm_rollout_params* params,
                            double* fitness, int32_t* trades, void* stream);

/* Same call with HOST pointers everywhere (genomes / master in, fitness / trades out): uploads,
 * runs, downloads and synchronises.  This is the end-to-end entry the Python
 * evaluate_individual / DRLEngine shims use when handed CPU tensors. */
int sgmm_rollout_population_host(const sgmm_bundle* bundle, const sgmm_population* mm,
                                 const sgmm_population* adv, const sgmm_rollout_params* params,
                                 double* fitness, int32_t* trades, void* stream);

/* Pipelined variant of the host-buffer entry for callers that evaluate batch after batch (a population service, or
 * independent populations such as a phi sweep): enqueues H2D + kernel + D2H of this batch on one of two internal streams
 * of the bundle and returns at once, so the upload of batch k+1 overlaps the kernel of batch k.  The HOST buffers
 * (genomes in, fitness / trades out; pinned memory for true overlap) must stay untouched until sgmm_rollout_wait(ticket)
 * returns.  At most two batches are in flight: a third call first waits for the oldest.  Same arguments otherwise. */
int sgmm_rollout_population_host_async(const sgmm_bundle* bundle, const sgmm_population* mm,
                                       const sgmm_population* adv, const sgmm_rollout_params* params,
                                       double* fitness, int32_t* trades, int32_t* ticket);
int sgmm_rollout_wait(const sgmm_bundle* bundle, int32_t ticket);

/* Audit variant of the tensor-core paths (hidden = 32 or 256, SGMM_PRECISION_BF16; F32 and EXACT are refused with
 * SGMM_ERR_INVALID): same kernel, plus
 *   raw_table  DEVICE float[count][T][5][2]  policy outputs for every (bar, inventory -2..2)
 *   act_trace  DEVICE int32[count][T][2]     the offsets actually taken along the walked trajectory
 * (either may be NULL).  Used to state the bf16 tolerance against the fp32 oracle and to replay the
 * taken actions through the oracle's env bit for bit. */
int sgmm_rollout_spec256_audit(const sgmm_bundle* bundle, const sgmm_population* mm,
                               const sgmm_rollout_params* params, double* fitness, int32_t* trades,
                               float* raw_table, int32_t* act_trace, void* stream);
/* The same with an adversary population (hidden = 32 or 256; adv may be NULL): act_trace holds the market maker's offsets
 * BEFORE the adversary's displacement (the recorder's off_a / off_b, Env/recorder.py:12), so that replaying them through
 * the reference's env together with the adversary genome reproduces the episode.  At hidden = 256 with an adversary the
 * rollout runs in batches in the bundle's code buffer, like an SGMM_PRECISION_EXACT rollout at H = 256. */
int sgmm_rollout_tc_audit(const sgmm_bundle* bundle, const sgmm_population* mm, const sgmm_population* adv,
                          const sgmm_rollout_params* params, double* fitness, int32_t* trades,
                          float* raw_table, int32_t* act_trace, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Per-step trace of ONE individual: the recorder row contract (Env/recorder.py:8-36,
 * main.py:74-90).  Every pointer is a DEVICE array of length T and may be NULL.
 * forced_actions (DEVICE int32[T,2], may be NULL) replaces the policy: teacher-forced replay of
 * recorded actions through the step core (bit-exact integer work given identical actions).
 * hidden = 32 or 256, both in SGMM-F32 order (H = 256: the exact policy table of sgmm_exact256.cu first, then the same
 * trace kernel; it uses the bundle's code buffer like an H = 256 population rollout).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t* off_a; int32_t* off_b;      /* MM action (before the adversary's displacement)      */
    int32_t* adv_a; int32_t* adv_b;      /* adversary displacement, 0 when off                   */
    int32_t* fill_buy; int32_t* fill_sell;
    int32_t* inventory;                  /* post-step                                            */
    double* cash; double* reward; double* pnl_reward; double* inventory_reward; double* fee_paid;
    float* raw_a; float* raw_b;          /* policy outputs before x5 and rounding                */
    /* the recorder's DERIVED columns (Env/recorder.py:45-51), computed in the same kernel pass: the two running sums
     * are sequential fp64 sums in bar order, exactly what pandas' cumsum does */
    double* spread;                      /* ask - bid                                            */
    double* wealth;                      /* cash + inventory * mid                               */
    double* cum_reward;                  /* reward.cumsum()                                      */
    int32_t* skew;                       /* off_b - off_a                                        */
    double* cum_fees;                    /* fee_paid.cumsum()                                    */
    double* unrealized_pnl;              /* inventory * mid     (realized_pnl is the cash column) */
} sgmm_trace;

int sgmm_rollout_trace(const sgmm_bundle* bundle, const float* mm_genome, int32_t hidden,
                       const float* adv_genome, const int32_t* forced_actions,
                       const sgmm_rollout_params* params, const sgmm_trace* trace,
                       double* fitness, int32_t* trades, void* stream);

/* Recorder traces of a whole population in one call (a backtest of many agents on one bundle: the top children of a
 * generation, several checkpoints, a phi / fee sweep, market maker and adversary pairs side by side).
 *   mm     the population as for sgmm_rollout_population: explicit genomes or seeded children (genomes == NULL: master +
 *          sigma * Philox from first_index on); hidden = 32 or 256.  adv may be NULL; otherwise adv->count == mm->count.
 *   trace  each non-NULL column is a DEVICE array [mm->count][T], row-major; row i holds exactly what sgmm_rollout_trace
 *          writes for individual i alone.  NULL columns are not written (trace itself may be NULL), and the work only they
 *          need is skipped.
 *   fitness / trades  DEVICE [mm->count], always written: bit-identical to the exact rollout (sgmm_rollout_population with
 *          SGMM_PRECISION_F32 at hidden 32, SGMM_PRECISION_EXACT at hidden 256).
 * The trace is in SGMM-F32 order whatever the width: params->precision must be SGMM_PRECISION_F32 or SGMM_PRECISION_EXACT
 * (BF16 / TF32 / F16: SGMM_ERR_UNSUPPORTED).  count == 0 writes nothing.  The raw policy table of a batch (40 B per
 * individual and bar, plus 269 KB per seeded or unaligned genome at hidden 256) lives in the bundle's code buffer, in batches
 * under SGMM_EXACT256_BATCH_BYTES: calls on one bundle must be ordered, and the first call of a size must not run under a
 * stream capture (as for sgmm_rollout_population above). */
int sgmm_rollout_trace_population(const sgmm_bundle* bundle, const sgmm_population* mm, const sgmm_population* adv,
                                  const sgmm_rollout_params* params, const sgmm_trace* trace,
                                  double* fitness, int32_t* trades, void* stream);

/* Inventory-table policies (benchmarks FOIC / GLFT, Env/benchmarks.py:3-40 driven by main.py:99-132):
 * the action at bar t is table[t][inv+2][{a,b}] (DEVICE int32[T,5,2]); same step core, same trace. */
int sgmm_rollout_table(const sgmm_bundle* bundle, const int32_t* table, const sgmm_rollout_params* params,
                       const sgmm_trace* trace, double* fitness, int32_t* trades, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Scalar env: FTPEnv.step / reset (Env/market_env.py:8-67) for the per-bar Python loops of the
 * blind test / backtest (pipeline/agent_trainer.py:144-153, pipeline/evaluator.py:25-37).
 * Host-side instantiation of the same step-core header the kernels use.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    double phi, tick_size, fee_rate;
    int64_t inventory;
    double cash;
    int64_t i_max, i_min;
} sgmm_env_state;

typedef struct {
    double reward, pnl_reward, inventory_reward, fee_paid;
    int32_t fill_buy, fill_sell;
} sgmm_step_info;

int sgmm_env_init(sgmm_env_state* e, double phi, double tick_size, double fee_rate);
int sgmm_env_step_host(sgmm_env_state* e, const int64_t action[2], const int64_t* adv_action,
                       double mid_next, double best_ask, double best_bid,
                       double buy_max, double sell_min, sgmm_step_info* info);
/* The same step with REAL-valued offsets: Env/market_env.py:23,30-31 uses the caller's offsets as given, so an unrounded
 * benchmark offset (e.g. GLFT's 1.7 ticks before rounding, Env/benchmarks.py) quotes at 1.7 ticks.  Identical to
 * sgmm_env_step_host for integral offsets. */
int sgmm_env_step_host_real(sgmm_env_state* e, const double action[2], const int64_t* adv_action,
                            double mid_next, double best_ask, double best_bid,
                            double buy_max, double sell_min, sgmm_step_info* info);

/* ---------------------------------------------------------------------------------------------
 * Device-side (1,lambda) evolution: NeuroEvolution.ask/tell + the generation loop of
 * DRLEngine.train (models/model.py:59-76, Env/drl_engine.py:92-171) with no host round trip:
 *   ask      children are regenerated from (master, sigma, seed, generation, index) in-kernel
 *   evaluate population rollout on the train bundle (adversary fused when use_arl)
 *   tell     argmax (first maximum) -> master <- best child; adversary: argmax of -fitness
 *   validate rollout of the new master on the val bundle, adversary off (:129-140)
 *   select   keep-best-on-validation snapshot (:144-150), sigma *= 0.5 after `patience`
 *            non-improving generations (:155-160), history append (:163-167)
 * ------------------------------------------------------------------------------------------- */
typedef struct sgmm_ga sgmm_ga;

typedef struct {
    int32_t hidden;           /* H */
    int32_t use_arl;          /* co-evolve the adversary (Env/drl_engine.py:75,80-81)            */
    int64_t pop_size;         /* GLOBAL lambda (models/model.py:60)                              */
    int64_t shard_first;      /* this rank evaluates children [shard_first, shard_first+shard_count) */
    int64_t shard_count;
    int64_t shard_stride;     /* 0 = unsharded (one rank owns the population); else the population is cut into */
                              /* blocks of shard_stride = ceil(pop_size / ranks) individuals, shard_first is a */
                              /* multiple of it and shard_count <= it (the last block may be short or empty)   */
    float sigma;              /* sigma_0 = 0.05 (models/model.py:61)                             */
    int32_t patience;         /* 15 (Env/drl_engine.py:155)                                      */
    double phi, fee_rate;
    uint64_t seed;
    int32_t max_generations;  /* history capacity                                                */
    int32_t precision;        /* SGMM_PRECISION_* of the POPULATION evaluation (0 = F32, bit-exact;  */
                              /* BF16 / TF32 / F16 = tensor-core rollout; EXACT = F32 at H=32).      */
                              /* hidden = 32: the validation rollout of the best child always runs   */
                              /* the exact F32 kernel.  hidden = 256 (BASELINE config 4): with a     */
                              /* tensor-core precision population AND validation run spec256_kernel; */
                              /* use_arl needs BF16 (the population's q tables walked by the exact   */
                              /* 20-state walk; validation stays without adversary).  With EXACT     */
                              /* both run the bit-exact H=256 path (sgmm_exact256.cu), use_arl       */
                              /* allowed.  F32 is refused at H=256.                                  */
} sgmm_ga_config;

typedef struct {
    int32_t generation;       /* generations completed                                           */
    int32_t stale;            /* non-improving generations since last improvement / decay        */
    float sigma, adv_sigma;
    double best_val;
    int64_t last_best_index;  /* global index of the last generation's best child               */
} sgmm_ga_status;

/* mm_master / adv_master: HOST float[G] / float[1250] initial masters (adv may be NULL unless use_arl) */
int sgmm_ga_create(sgmm_ga** out, const sgmm_ga_config* cfg, const float* mm_master,
                   const float* adv_master, int device, void* stream);
int sgmm_ga_destroy(sgmm_ga* ga);
/* The population's results live in ONE rank-blocked DEVICE buffer, so that a sharded generation needs a single
 * collective:   block r = { double fitness[stride]; int32_t trades[stride]; pad to 16 B }   (block_bytes each)
 * holds individuals [r*stride, (r+1)*stride), stride = shard_stride (or pop_size when unsharded: one block).
 * fitness_slice / trades_slice point into this rank's block (my_block = shard_first / stride); sgmm_ga_evaluate
 * writes them, sgmm_ga_select reads all n_blocks blocks.  A multi-GPU caller all-gathers its block IN PLACE
 * (ncclAllGather(base + my_block*block_bytes, base, block_bytes, ncclChar) -- torch: all_gather_into_tensor on uint8
 * views) between the two phases: one collective per generation, fitness and trade counts together (INTEGRATION.md).
 * Any output pointer may be NULL. */
int sgmm_ga_buffers(sgmm_ga* ga, double** fitness_slice, int32_t** trades_slice, void** gather_base,
                    int64_t* block_bytes, int32_t* n_blocks, int32_t* my_block);
/* phase 1: ask + evaluate this rank's shard on `train` */
int sgmm_ga_evaluate(sgmm_ga* ga, const sgmm_bundle* train, void* stream);
/* phase 2: tell + validate on `val` + keep-best + sigma decay + history; advances the generation */
int sgmm_ga_select(sgmm_ga* ga, const sgmm_bundle* val, void* stream);
/* both phases back to back (single rank) */
int sgmm_ga_generation(sgmm_ga* ga, const sgmm_bundle* train, const sgmm_bundle* val, void* stream);
/* synchronising read-backs (HOST pointers) */
int sgmm_ga_status_host(sgmm_ga* ga, sgmm_ga_status* status, void* stream);
int sgmm_ga_master_host(sgmm_ga* ga, float* mm_master, float* adv_master, float* best_val_master,
                        void* stream);
/* history columns of Env/drl_engine.py:86-89,163-167; each HOST array of capacity n, may be NULL */
int sgmm_ga_history_host(sgmm_ga* ga, int32_t n, double* train_f, double* val_f,
                         int32_t* train_trades, int32_t* val_trades, float* sigma, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Upstream of the rollout: the per-day window loop of load_signals_bundle
 * (pipeline/agent_trainer.py:47-73).  Inputs are one day's event frame columns (loader2.event_df:
 * askprice1, bidprice1, p_buy_max, p_sell_min; n_events rows, NaN allowed in the last two) and
 * n_signals = min(len(s1_pred), len(s2_pred)) (:47).  The events are sampled every event_step rows
 * (:49), the last n_signals samples are kept, and for each consecutive pair the outputs are
 *   buy_max / sell_min  NaN-skipping max / min over the INCLUSIVE window between the two samples (:54-59)
 *   best_ask / best_bid of the current sample (:70-71),  mid_next = (ask + bid) / 2 of the next (:73)
 * n_signals - 1 values each (none if n_signals <= 1).  SGMM_ERR_INVALID if n_signals exceeds the
 * number of sampled events ceil(n_events / event_step).  z-normalisation and train_stats stay on the
 * host with the caller's own numpy expression (they are float32 pairwise reductions of numpy).
 * ------------------------------------------------------------------------------------------- */
int sgmm_bundle_windows(int64_t n_events, const double* askprice1, const double* bidprice1,
                        const double* p_buy_max, const double* p_sell_min, int64_t event_step, int64_t n_signals,
                        double* mid_next, double* best_ask, double* best_bid, double* buy_max, double* sell_min,
                        void* stream);                                   /* DEVICE pointers, no sync */
int sgmm_bundle_windows_host(int64_t n_events, const double* askprice1, const double* bidprice1,
                             const double* p_buy_max, const double* p_sell_min, int64_t event_step, int64_t n_signals,
                             double* mid_next, double* best_ask, double* best_bid, double* buy_max, double* sell_min,
                             int device, void* stream);                   /* HOST pointers, synchronises */

/* ---------------------------------------------------------------------------------------------
 * Downstream of the rollout: StrategyAnalytics.summary_dict (analytics/mm_analyzer.py:5-56) for a
 * batch of n_traces traces of n_steps rows each (row-major [n_traces, n_steps]):
 *   out[b] = { Total PnL, MAP (Risk), PnLMAP (Eff), Max DD, Sharpe, Trades }        float64[6]
 * wealth may be NULL, in which case it is derived as cash + inventory * mid (Env/recorder.py:46) with
 * mid[n_steps] shared by all traces (the sgmm_rollout_trace outputs plug in directly).
 * scratch: DEVICE float64[n_traces, n_steps] workspace.  Reductions follow pandas / numpy's pairwise
 * float64 summation order, so the Sharpe ratio is bit-identical to the reference's.
 * ------------------------------------------------------------------------------------------- */
int sgmm_trace_analytics(int64_t n_traces, int64_t n_steps, const double* wealth, const double* cash,
                         const double* mid, const int32_t* inventory, const uint8_t* is_trade,
                         double* scratch, double* out, void* stream);    /* DEVICE pointers, no sync */
int sgmm_trace_analytics_host(int64_t n_traces, int64_t n_steps, const double* wealth, const int32_t* inventory,
                              const uint8_t* is_trade, double* out, int device, void* stream);   /* HOST pointers */

/* sizeof() of the public structs as this library was compiled, for foreign-function bindings to verify their
 * mirrors: which = 0 sgmm_population, 1 sgmm_rollout_params, 2 sgmm_trace, 3 sgmm_env_state, 4 sgmm_step_info,
 * 5 sgmm_ga_config, 6 sgmm_ga_status; negative for an unknown index. */
int sgmm_abi_sizeof(int which);

/* ---------------------------------------------------------------------------------------------
 * Measurement helper: sustained FP32 FFMA throughput of the device (TFLOP/s), the denominator of
 * the H=32 roofline (SURVEY.md section 8d asks for a measured FFMA peak).
 * ------------------------------------------------------------------------------------------- */
int sgmm_measure_fp32_peak(int device, double* tflops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SGMM_H */
