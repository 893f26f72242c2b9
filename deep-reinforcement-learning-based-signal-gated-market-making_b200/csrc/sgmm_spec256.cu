// sgmm_spec256.cu -- H = 256 policy rollout on the 5th-generation tensor cores (tcgen05 + TMEM).
//
// BASELINE.json config 4 ("wider MLP hidden sizes (256x256) on tensor cores").  Per individual the
// sequential rollout is a chain of 256x256 GEMVs -- no batch dimension, the tensor cores would
// idle.  The inventory is a 5-valued integer ({-2..2}, Env/market_env.py:14-15,34-35), so the
// action at bar t is a function of (t, inv) only (SURVEY.md 7.3): evaluate the policy for ALL five
// inventories of every bar (time-parallel speculation) and the hidden layer becomes a real GEMM
//     D[(t,inv), j] = sum_k h1[(t,inv), k] * W2[j, k]        M = 5*T rows, N = K = 256
// followed by a trivially cheap walk of the 5-state automaton.  5x the hidden-layer FLOPs, on a
// pipe ~30x faster than the FP32 cores, and no step-to-step latency chain.
//
// One persistent CTA per SM, one individual at a time, warp-specialised.  Layers 2 AND 3 run on the tensor
// cores; the CUDA cores only convert the accumulator in place (the structure of sgmm_tc32.cu):
//   warps 0-3   epilogue: per tile, E3 of the previous tile then E2 of this one
//                 E2      : tcgen05.ld.pack::16b of D2 (lane = row, f16 accumulators: two columns per register),
//                           bias + ReLU in one fma.rn.relu.f16x2 per pair, tcgen05.st of A3 IN PLACE (columns 0..127
//                           of the same TMEM buffer)
//                 E3      : tcgen05.ld of D3 (4 columns: W3 hi + lo), +b3, x5 + round-half-even, and the
//                           SPECULATIVE env step of the row's (bar, inventory): fills, next inventory, fp64
//                           reward (Env/market_env.py:30-58) -> reward table + 1-byte next-state table
//   warps 4-11  producer: layer 1 (3->256) in fp32 SGMM order for the 5 inventories of 25 bars,
//                         cvt.rn.relu.f16x2, 128B-swizzled K-major A tile (4 k-blocks of 16 KB, ring);
//                         two warps per k-block, so the four k-blocks of a tile are produced in parallel
//                         (a serial producer made the tile period 4 x its k-block latency: 3 900 of 5 400 cycles)
//   warp  12    MMA     : converged warp, one elected lane issues BOTH GEMMs in one stream:
//                         L2 tcgen05.mma.cta_group::1.kind::f16 (M=128, N=256, K=16) x16 per tile, A and B from shared
//                         memory, D2 in TMEM (2 buffers x 256 columns, f16 accumulators);
//                         L3 (M=128, N=16, K=16) x16 of the PREVIOUS tile slotted between the k-blocks of L2: A3 read
//                         FROM TENSOR MEMORY, B3 = W3 hi / lo rows from shared memory, D3 (fp32) into columns 128..143
//                         of the same buffer (dead after E2)
//   warp  13    walker  : two-phase walk of the tile (automaton on the byte table, then the fp64 reward sum in
//                         reference order), trades; fitness / trade count out (Env/drl_engine.py:54-67)
// W2 (f16, 128 KB, swizzled K-major B operand) stays resident in shared memory for the episode.
//
// With the adversary (q-table mode, QTAB = true) the next state of a bar depends on the previous bar's fills as well, a
// 20-state automaton (sgmm_one.cu, Walk20): E3 writes q = raw*5 of every (bar, inventory) row to global memory instead
// of step codes, the walker warp idles, and walk_account_kernel<Walk20> walks the table afterwards (launch_spec256_adv).
//
// Precision: h1, W2 and the layer-2 accumulator are f16 (11 significand bits), the output layer accumulates in fp32;
// tests/test_gpu_spec256.py states the tolerance against the fp32 oracle (0.05 tick; measured 0.008), checks that no
// rounding flips where the oracle's margin exceeds it, and checks that GIVEN the kernel's actions
// every integer and fp64 quantity is bit-identical to the oracle (teacher-forced replay).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdio>
#include "sgmm_internal.h"
#include "sgmm_rng.cuh"
#include "sgmm_step_core.h"

namespace sgmm {

namespace s256 {
#ifdef SGMM_SPEC256_TRACE
#define TR(ev) do { if (blockIdx.x == 0 && gt == 0 && it >= 64 && it < 72 && lane == 0) sm.trace[it - 64][ev] = clock64(); } while (0)
#else
#define TR(ev) do { } while (0)
#endif

constexpr int H = 256;
constexpr int TILE_ROWS = 128;
constexpr int TILE_BARS = 25;                 // 25 bars x 5 inventories = 125 rows (+3 idle rows)
constexpr int KBLK = 64;                      // bf16 elements per 128-byte swizzle row
constexpr int NKB = H / KBLK;                 // 4 k-blocks
constexpr int UMMA_K = 16;
constexpr int NUM_EPI_WARPS = 4, NUM_PROD_WARPS = 8;      // epilogue warps 0-3 (one per TMEM lane quarter) run E3(i-1) then E2(i)
constexpr int WARP_MMA = 12, WARP_WALK = 13;
constexpr int NUM_THREADS = 448;
constexpr int L3_SLOT = 2;                    // layer 3 of the previous tile is issued before this k-block of layer 2
constexpr int B3_BYTES = 16 * H * 2;          // W3 hi (rows 0,1) and bf16 residual (rows 2,3), canonical K-major layout
constexpr uint32_t C_D3 = 128;                // D3 lives in columns 128..143 of the buffer (free once E2 has read D2)
constexpr uint32_t TMEM_COLS = 512;
constexpr int64_t G = (int64_t)H * H + 7 * H + 2;       // 67330

// One 25-bar tile of the walk through the table (the same two-phase walk as sgmm_tc32.cu):
//   phase A: the 5-state automaton alone -- a 2-instruction chain per bar (byte `w` of the bar's 8-byte record:
//            next | traded << 3), its loads independent of the chain;
//   phase B: the step codes of the visited rows go to global memory in bar order; the fp64 accounting (rewards,
//            reference-order sum, trade count) is sgmm_account.cu's, AFTER this kernel: an FP64 instruction issued
//            while tcgen05.mma executes waits ~740 cycles instead of 9 (tools/walk_bench.cu).
// (A walk that chased one 32-byte entry per bar -- load, then the next address from the loaded inventory -- cost 170
//  cycles per bar and was THE bottleneck of this kernel: 4 200 of the tile's 4 200 cycles, profiles/r1_spec256_trace.txt.)
template <bool FULL>
__device__ __forceinline__ void walk_tile(const uint8_t* nb, const uint64_t* cb, int n, int& iv, uint64_t* out)
{
    uint32_t ivs[TILE_BARS];
    uint32_t w = (uint32_t)iv;
#pragma unroll
    for (int s = 0; s < TILE_BARS; ++s) {
        ivs[s] = w;
        if (FULL || s < n) {
            const uint2 x = *reinterpret_cast<const uint2*>(nb + s * 8);
            w = __byte_perm(x.x, x.y, w) & 7u;
        }
    }
    iv = (int)w;
#pragma unroll
    for (int s = 0; s < TILE_BARS; ++s)
        if (FULL || s < n) __stcs(out + s, cb[s * 5 + ivs[s]]);          // the visited row's step code (sgmm_account.cu)
}

struct Smem {
    uint8_t b_tile[NKB][H * 128];              // W2 bf16, [k-block][n][64] swizzled, 128 KB
    uint8_t a_tile[NKB][TILE_ROWS * 128];      // h1 bf16, [k-block][row][64] swizzled, 64 KB
    uint8_t b3_tile[B3_BYTES];                 // layer-3 B operand (no swizzle: 8 x 16-byte core matrices)
    float w1x[H], w1y[H], w1i[H], b1[H], b2[H];
    uint32_t b2h[H / 2];                       // b2 as f16 pairs (F16 build: added by the epilogue's HFMA2.RELU)
    float b3[4];
    uint64_t tab_c[2][TILE_ROWS];              // step code of (bar, inventory) rows: offsets, fills, |inv'| (sgmm_account.cu)
    alignas(8) uint8_t tab_n[2][TILE_BARS * 8]; // next inventory index | traded << 3, 8 bytes per bar
    int32_t tab_k[2][TILE_ROWS][2];            // quantised offsets of the row (audit: act_trace)
    // d_full: L2 committed (D2 complete); a3_ready: E2 wrote A3; l3_done: L3 committed (D3 complete);
    // d_empty: E3 has read D3, the buffer may take the next D2
    uint64_t a_full[NKB], a_empty[NKB], d_full[2], a3_ready[2], l3_done[2], d_empty[2], t_full[2], t_empty[2];
    uint32_t tmem_base;
    uint32_t pad;
#ifdef SGMM_SPEC256_TRACE
    long long trace[8][16];
#endif
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE_%=;\n"
        "bra LAB_WAIT_%=;\n"
        "LAB_DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start>>4 | [16,30) LBO>>4 (unused for swizzled K-major) | [32,46) SBO>>4 = 1024 B (8 rows)
//   [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr)
{
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c=f32 (bit 4), a=b=bf16 (bits 7,10), K-major both,
// n_dim = N>>3 at [17,23), m_dim = M>>4 at [24,29)
// F16 = true: f16 operands and an F16 accumulator for layer 2 (c format 0, a/b format 0).  One f16 per TMEM column,
// read back two columns per register (.pack::16b): half the tensor-memory read traffic of the epilogue, bias + ReLU in
// ONE HFMA2.RELU per pair and no conversion; f16 keeps 11 significand bits against bf16's 8.  Layer 3 accumulates in fp32.
constexpr bool F16 = true;
constexpr uint32_t IDESC = (F16 ? 0u : ((1u << 4) | (1u << 7) | (1u << 10))) | ((uint32_t)(H >> 3) << 17) | ((uint32_t)(TILE_ROWS >> 4) << 24);

__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate) : "memory");
}
// layer 3: A operand from tensor memory, B (no swizzle) from shared memory, N = 16
constexpr uint32_t IDESC_L3 = (1u << 4) | (F16 ? 0u : ((1u << 7) | (1u << 10))) | ((uint32_t)(16 >> 3) << 17) | ((uint32_t)(TILE_ROWS >> 4) << 24);
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(IDESC_L3), "r"(accumulate) : "memory");
}
// K-major SWIZZLE_NONE descriptor (checked by tools/tc32_unit.cu): LBO = distance of the two 16-byte k-chunks of a
// K=16 step, SBO = distance of 8-row groups
__device__ __forceinline__ uint64_t make_desc_ns(uint32_t saddr, uint32_t lbo, uint32_t sbo)
{
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
__device__ __forceinline__ uint32_t canon(int r, int k, int K) { return (uint32_t)(((r >> 3) * (K >> 3) + (k >> 3)) * 128 + (r & 7) * 16 + (k & 7) * 2); }
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&v)[4])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
                 "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
__device__ __forceinline__ uint16_t bf16_bits(float x) { return __bfloat16_as_ushort(__float2bfloat16_rn(x)); }

__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// two fp32 -> packed bf16x2 with ReLU; `lo` lands in the low half (lower address)
__device__ __forceinline__ uint32_t pack_relu_bf16(float lo, float hi)        // (operand type of the build: bf16 or f16)
{
    uint32_t r;
    if (F16) asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    else asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi)
{
    uint32_t r;
    if (F16) asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ float op_round(float x) { return F16 ? __half2float(__float2half_rn(x)) : bf16_round(x); }
__device__ __forceinline__ uint16_t op_bits(float x) { return F16 ? __half_as_ushort(__float2half_rn(x)) : bf16_bits(x); }
// 32 columns of 16-bit accumulators -> 16 registers of f16x2 pairs (column 2c low, 2c+1 high)
__device__ __forceinline__ void tmem_ld32_pack16(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.pack::16b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ uint32_t hfma2_relu(uint32_t a, uint32_t b, uint32_t c)   // relu(a * b + c) on f16 pairs
{
    uint32_t r;
    asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ uint32_t bias_relu_f16x2(uint32_t x, uint32_t b)  // relu(x * 1 + b) on f16 pairs (HFMA2.RELU)
{
    uint32_t r;
    asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(x), "r"(0x3C003C00u), "r"(b));
    return r;
}
// byte offset of 16-byte chunk `c` (8 bf16) of row `r` inside a [rows][128 B] SWIZZLE_128B slab
__device__ __forceinline__ uint32_t swz(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }

struct Args {
    const BarSig* sig; const BarPx* px; uint64_t* codes; int64_t T;
    double tick, phi, fee;
    PopArgs mm;
    double* fitness; int32_t* trades;
    float* raw_table;        // optional audit output [P][T][5][2]
    int32_t* act_trace;      // optional audit output [P][T][2] : actions actually taken
    float2* qtab;            // q-table mode: q = raw*5 of every (bar, inventory) [P][T][5] (Walk20's table)
};

template <bool FEE, bool QTAB = false>
__global__ void __launch_bounds__(NUM_THREADS, 1) spec256_kernel(const Args a)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // SWIZZLE_128B operands need 1024-byte aligned slabs (descriptor base_offset = 0)
    const uint32_t misalign = smem_u32(smem_raw) & 1023u;
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw + ((1024u - misalign) & 1023u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t T = a.T;
    const int64_t ntiles = (T + TILE_BARS - 1) / TILE_BARS;

    if (tid == 0) {
        for (int i = 0; i < NKB; ++i) { mbar_init(&sm.a_full[i], NUM_PROD_WARPS / NKB); mbar_init(&sm.a_empty[i], 1); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&sm.d_full[i], 1); mbar_init(&sm.a3_ready[i], 4); mbar_init(&sm.l3_done[i], 1);
            mbar_init(&sm.d_empty[i], 4);
            mbar_init(&sm.t_full[i], 4); mbar_init(&sm.t_empty[i], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == WARP_MMA) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < B3_BYTES / 16; i += NUM_THREADS) reinterpret_cast<uint4*>(sm.b3_tile)[i] = make_uint4(0, 0, 0, 0);
    // rows 125..127 of the A tile are never produced: keep them finite
    for (int i = tid; i < NKB * TILE_ROWS * 128 / 16; i += NUM_THREADS)
        reinterpret_cast<uint4*>(&sm.a_tile[0][0])[i] = make_uint4(0, 0, 0, 0);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sm.tmem_base;

    const PopArgs pop = resolve(a.mm);           // GA: sigma / generation come from device scalars
    uint32_t gt = 0;                               // tiles processed so far by this CTA (pipeline phase source)

    for (int64_t ind = blockIdx.x; ind < pop.count; ind += gridDim.x) {
        // ---------------- stage the individual's weights (all warps) ----------------------------
        {
            GenomeSource src;
            src.seeded = (pop.genomes == nullptr);
            src.row = src.seeded ? pop.master : pop.genomes + ind * G;
            src.sigma = pop.sigma; src.seed = pop.seed; src.generation = pop.generation;
            src.individual = (uint64_t)(pop.first_index + ind);
            const int64_t offW2 = 4 * H;                      // W1[H,3] | b1[H] | W2[H,H] | b2 | W3[2,H] | b3[2]
            for (int q = tid; q < H * H / 8; q += NUM_THREADS) {        // 8 consecutive k of one row j
                const int j = q / (H / 8), kc = q % (H / 8);           // kc: 16-byte chunk along k (0..31)
                float v[4], w[4];
                src.at4(offW2 + (int64_t)j * H + kc * 8, v);
                src.at4(offW2 + (int64_t)j * H + kc * 8 + 4, w);
                uint4 o;
                o.x = pack_bf16(v[0], v[1]); o.y = pack_bf16(v[2], v[3]);
                o.z = pack_bf16(w[0], w[1]); o.w = pack_bf16(w[2], w[3]);
                *reinterpret_cast<uint4*>(&sm.b_tile[kc >> 3][swz(j, kc & 7)]) = o;
            }
            for (int j = tid; j < H; j += NUM_THREADS) {
                sm.w1x[j] = src.at(3 * j); sm.w1y[j] = src.at(3 * j + 1); sm.w1i[j] = src.at(3 * j + 2);
                sm.b1[j] = src.at(3 * H + j);
                sm.b2[j] = src.at(4 * H + (int64_t)H * H + j);
            }
            for (int j = tid; j < H / 2; j += NUM_THREADS)
                sm.b2h[j] = pack_bf16(src.at(4 * H + (int64_t)H * H + 2 * j), src.at(4 * H + (int64_t)H * H + 2 * j + 1));
            for (int q = tid; q < 2 * H; q += NUM_THREADS) {                  // W3[o, k]: row o = bf16(w), row o+2 = bf16 residual
                const int o = q / H, k = q % H;
                const float w = src.at(5 * H + (int64_t)H * H + q);
                const float h = op_round(w), m = op_round(__fadd_rn(w, -h));
                *reinterpret_cast<uint16_t*>(&sm.b3_tile[canon(o, k, H)]) = op_bits(h);
                *reinterpret_cast<uint16_t*>(&sm.b3_tile[canon(o + 2, k, H)]) = op_bits(m);
            }
            if (tid < 2) sm.b3[tid] = src.at(7 * H + (int64_t)H * H + tid);
        }
        fence_proxy_async();                       // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncthreads();

        if (warp < NUM_EPI_WARPS) {
            // =========================== EPILOGUE : E3 of tile it-1, then E2 of tile it =================
            const int quarter = warp & 3;
            const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16);
            const int row = quarter * 32 + lane;
            const int tl = row / 5, iv = row % 5;          // bar within the tile, inventory index (inv+2)
            auto e2 = [&](int64_t it) {                    // D2 -> +b2 -> relu -> bf16 -> A3 in place
                const uint32_t g = gt + (uint32_t)it, buf = g & 1u, use = g >> 1;
                mbar_wait(&sm.d_full[buf], use & 1u);
                tc_fence_after();
                if (warp == 0) TR(3);
                const uint32_t tbase = lane_addr + buf * 256u;
                if (F16) {
                    uint32_t h[2][16];
                    tmem_ld32_pack16(tbase, h[0]);
#pragma unroll
                    for (int cc = 0; cc < H / 32; ++cc) {
                        tmem_ld_wait();                                    // chunk cc has landed
                        if (cc + 1 < H / 32) tmem_ld32_pack16(tbase + (uint32_t)((cc + 1) * 32), h[(cc + 1) & 1]);   // prefetch
                        const uint32_t* w = h[cc & 1];
                        uint32_t p[16];
#pragma unroll
                        for (int c = 0; c < 16; c += 4) {
                            const uint4 bb = *reinterpret_cast<const uint4*>(&sm.b2h[cc * 16 + c]);
                            p[c] = bias_relu_f16x2(w[c], bb.x); p[c + 1] = bias_relu_f16x2(w[c + 1], bb.y);
                            p[c + 2] = bias_relu_f16x2(w[c + 2], bb.z); p[c + 3] = bias_relu_f16x2(w[c + 3], bb.w);
                        }
                        tmem_st16(tbase + (uint32_t)(cc * 16), p);        // writes trail reads (see below)
                    }
                } else {
                    uint32_t v[2][32];
                    tmem_ld32(tbase, v[0]);
#pragma unroll
                    for (int cc = 0; cc < H / 32; ++cc) {
                        tmem_ld_wait();                                        // chunk cc has landed
                        if (cc + 1 < H / 32) tmem_ld32(tbase + (uint32_t)((cc + 1) * 32), v[(cc + 1) & 1]);   // prefetch
                        const uint32_t* w = v[cc & 1];
                        uint32_t p[16];
#pragma unroll
                        for (int c = 0; c < 32; c += 4) {
                            const float4 bb = *reinterpret_cast<const float4*>(&sm.b2[cc * 32 + c]);
                            const float2 x0 = __fadd2_rn(make_float2(__uint_as_float(w[c]), __uint_as_float(w[c + 1])), make_float2(bb.x, bb.y));
                            const float2 x1 = __fadd2_rn(make_float2(__uint_as_float(w[c + 2]), __uint_as_float(w[c + 3])), make_float2(bb.z, bb.w));
                            p[c >> 1] = pack_relu_bf16(x0.x, x0.y);
                            p[(c >> 1) + 1] = pack_relu_bf16(x1.x, x1.y);
                        }
                        // columns 16cc..16cc+15 were read (as part of chunk cc/2) before they are overwritten: writes trail reads
                        tmem_st16(tbase + (uint32_t)(cc * 16), p);
                    }
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.a3_ready[buf]);
                if (warp == 0) TR(4);
            };
            auto e3 = [&](int64_t it) {                    // D3 -> offsets -> speculative env step -> table
                const uint32_t g = gt + (uint32_t)it, buf = g & 1u, use = g >> 1;
                // bar data of this row's step: issued before the accumulator is ready (L2 latency hides behind the wait)
                const int64_t t = it * TILE_BARS + tl;
                const bool valid = (row < TILE_BARS * 5) && (t < T);
                const int64_t tc_ = valid ? t : 0;
                int2 kth = make_int2(0, 0);
                if (!QTAB && T > 0) kth = __ldg(reinterpret_cast<const int2*>(&a.sig[tc_].ka1));
                mbar_wait(&sm.l3_done[buf], use & 1u);
                tc_fence_after();
                if (warp == 0) TR(5);
                uint32_t v[4];
                tmem_ld4(lane_addr + buf * 256u + C_D3, v);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.d_empty[buf]);                // the buffer may take the next D2
                if (warp == 0) TR(6);
                const float ra = __fadd_rn(__fadd_rn(__uint_as_float(v[0]), __uint_as_float(v[2])), sm.b3[0]);   // W3 hi + lo, + b3
                const float rb = __fadd_rn(__fadd_rn(__uint_as_float(v[1]), __uint_as_float(v[3])), sm.b3[1]);
                const int ka = __float2int_rn(__fmul_rn(ra, 5.0f));          // drl_engine.py:39
                const int kb = __float2int_rn(__fmul_rn(rb, 5.0f));
                // speculative env step of (bar t, inventory iv-2)  (market_env.py:30-58)
                uint64_t code = 0; uint32_t nxt = (uint32_t)iv;
                if (valid) {
                    if constexpr (QTAB) {
                        // the row's q, as fl(raw*5) above; the 125 rows of a tile are contiguous: coalesced stores
                        a.qtab[((int64_t)ind * T + t) * 5 + iv] = make_float2(__fmul_rn(ra, 5.0f), __fmul_rn(rb, 5.0f));
                    } else {
                        // the INTEGER half of the env step (market_env.py:34-38, 45, 51); quotes, P&L and the penalty are
                        // fp64 and belong to the accounting pass
                        const int inv = iv - 2;
                        const bool fb = (inv < 2) && (kb < kth.y);               // :34,:37
                        const bool fs = (inv > -2) && (ka < kth.x);              // :35,:38
                        const int ninv = inv + (fb ? 1 : 0) - (fs ? 1 : 0);
                        code = (uint64_t)(uint32_t)(fs ? ka : SGMM_CODE_NOFILL) | ((uint64_t)(uint32_t)(fb ? kb : SGMM_CODE_NOFILL) << 32);
                        nxt = (uint32_t)(ninv + 2) | ((fb || fs) ? 8u : 0u);
                    }
                    if (a.raw_table) {
                        float* o = a.raw_table + (((int64_t)ind * T + t) * 5 + iv) * 2;
                        o[0] = ra; o[1] = rb;
                    }
                }
                if constexpr (QTAB) return;                // no tile table: t_full / t_empty stay untouched in this mode
                // publish the tile's table
                if (warp == 0) TR(13);
                mbar_wait(&sm.t_empty[buf], (use & 1u) ^ 1u);
                if (warp == 0) TR(14);
                if (row < TILE_BARS * 5) {
                    sm.tab_c[buf][row] = code;
                    sm.tab_n[buf][tl * 8 + iv] = (uint8_t)nxt;
                    if (a.act_trace) { sm.tab_k[buf][row][0] = ka; sm.tab_k[buf][row][1] = kb; }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.t_full[buf]);
                if (warp == 0) TR(7);
            };
            for (int64_t it = 0; it < ntiles; ++it) {
                if (it > 0) e3(it - 1);
                e2(it);
            }
            if (ntiles > 0) e3(ntiles - 1);
        } else if (warp < NUM_EPI_WARPS + NUM_PROD_WARPS) {
            // =========================== PRODUCER ==============================================
            // Two warps per k-block: the four k-blocks of a tile are produced IN PARALLEL, each pair waiting only
            // for its own slot (a ring of one tile: a serial producer made the tile period 4 x its k-block latency).
            const int pw = warp - NUM_EPI_WARPS;           // 0..7
            const int kb = pw >> 1;                        // this pair's k-block
            const int gtid = (pw & 1) * 32 + lane;         // 0..63 within the pair
            const int c = gtid & 7;                        // this thread's 16-byte chunk (8 k) of the k-block
            const int k0 = kb * KBLK + c * 8;
            // the thread's layer-1 weights are the same for every tile of the individual: registers
            float2 wx[4], wy[4], wi[4], bb[4];
            {
                const float4 p0 = *reinterpret_cast<const float4*>(&sm.w1x[k0]), p1 = *reinterpret_cast<const float4*>(&sm.w1x[k0 + 4]);
                wx[0] = make_float2(p0.x, p0.y); wx[1] = make_float2(p0.z, p0.w); wx[2] = make_float2(p1.x, p1.y); wx[3] = make_float2(p1.z, p1.w);
                const float4 q0 = *reinterpret_cast<const float4*>(&sm.w1y[k0]), q1 = *reinterpret_cast<const float4*>(&sm.w1y[k0 + 4]);
                wy[0] = make_float2(q0.x, q0.y); wy[1] = make_float2(q0.z, q0.w); wy[2] = make_float2(q1.x, q1.y); wy[3] = make_float2(q1.z, q1.w);
                const float4 r0 = *reinterpret_cast<const float4*>(&sm.w1i[k0]), r1 = *reinterpret_cast<const float4*>(&sm.w1i[k0 + 4]);
                wi[0] = make_float2(r0.x, r0.y); wi[1] = make_float2(r0.z, r0.w); wi[2] = make_float2(r1.x, r1.y); wi[3] = make_float2(r1.z, r1.w);
                const float4 s0 = *reinterpret_cast<const float4*>(&sm.b1[k0]), s1 = *reinterpret_cast<const float4*>(&sm.b1[k0 + 4]);
                bb[0] = make_float2(s0.x, s0.y); bb[1] = make_float2(s0.z, s0.w); bb[2] = make_float2(s1.x, s1.y); bb[3] = make_float2(s1.z, s1.w);
            }
            uint32_t wih[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) wih[p] = pack_bf16(wi[p].x, wi[p].y);
            uint8_t* slab = &sm.a_tile[kb][0];
            for (int64_t it = 0; it < ntiles; ++it) {
                const uint32_t g = gt + (uint32_t)it;
                const int64_t t0 = it * TILE_BARS;
                // the thread's (up to) four bars of this tile: tasks q = gtid + 64 m = (bar, chunk)
                float2 z[4];
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    const int tlm = (gtid >> 3) + 8 * m;
                    const int64_t t = t0 + tlm < T ? t0 + tlm : T - 1;
                    z[m] = (tlm < TILE_BARS) ? *reinterpret_cast<const float2*>(&a.sig[t].z1) : make_float2(0.f, 0.f);
                }
                // the slot: wait until the MMAs of the previous tile have consumed it
                if (g > 0) mbar_wait(&sm.a_empty[kb], (g - 1) & 1u);
                if (pw == 0) TR(9);
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    const int tlm = (gtid >> 3) + 8 * m;
                    if (tlm < TILE_BARS) {
                        float2 A[4];
#pragma unroll
                        for (int p = 0; p < 4; ++p)          // SGMM-F32 layer 1: b1, +W1[.,0] z1, +W1[.,1] z2
                            A[p] = __ffma2_rn(wy[p], make_float2(z[m].y, z[m].y), __ffma2_rn(wx[p], make_float2(z[m].x, z[m].x), bb[p]));
                        if (F16) {
                            // the bar part of layer 1 stays in fp32 (SGMM order) and is rounded ONCE to f16 pairs; the
                            // inventory term and the ReLU are one HFMA2.RELU per pair and row: no per-row conversion
                            // (cvt.rn.relu.f16x2.f32 per row kept the XU pipe at 129 %)
                            uint32_t Ah[4];
#pragma unroll
                            for (int p = 0; p < 4; ++p) Ah[p] = pack_bf16(A[p].x, A[p].y);
#pragma unroll
                            for (int iv = 0; iv < 5; ++iv) {
                                // inv / 2 as an f16 pair (drl_engine.py:35): -1, -0.5, 0, 0.5, 1
                                const uint32_t i2 = iv == 0 ? 0xBC00BC00u : iv == 1 ? 0xB800B800u : iv == 2 ? 0u : iv == 3 ? 0x38003800u : 0x3C003C00u;
                                uint4 o;
                                o.x = hfma2_relu(wih[0], i2, Ah[0]); o.y = hfma2_relu(wih[1], i2, Ah[1]);
                                o.z = hfma2_relu(wih[2], i2, Ah[2]); o.w = hfma2_relu(wih[3], i2, Ah[3]);
                                const int r = tlm * 5 + iv;
                                *reinterpret_cast<uint4*>(slab + swz(r, c)) = o;
                            }
                        } else {
    #pragma unroll
                            for (int iv = 0; iv < 5; ++iv) {
                                const float inv2 = (float)(iv - 2) * 0.5f;       // drl_engine.py:35
                                uint4 o;
                                float2 v0 = __ffma2_rn(wi[0], make_float2(inv2, inv2), A[0]);
                                float2 v1 = __ffma2_rn(wi[1], make_float2(inv2, inv2), A[1]);
                                float2 v2 = __ffma2_rn(wi[2], make_float2(inv2, inv2), A[2]);
                                float2 v3 = __ffma2_rn(wi[3], make_float2(inv2, inv2), A[3]);
                                o.x = pack_relu_bf16(v0.x, v0.y); o.y = pack_relu_bf16(v1.x, v1.y);
                                o.z = pack_relu_bf16(v2.x, v2.y); o.w = pack_relu_bf16(v3.x, v3.y);
                                const int r = tlm * 5 + iv;
                                *reinterpret_cast<uint4*>(slab + swz(r, c)) = o;
                            }
                        }
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.a_full[kb]);
                if (pw == 0) TR(10);
            }
        } else if (warp == WARP_MMA) {
            // =========================== MMA ISSUER (converged warp, one elected lane issues) ===========
            // ONE issue stream for both GEMMs: layer 3 of tile it-1 is slotted between the k-blocks of layer 2 of tile
            // it.  (With its own issuer warp the sixteen small layer-3 MMAs took turns with the big layer-2 MMAs of the
            // next tile, finished only when that tile did, and the buffer hand-back E3 -> d_empty -> next layer 2 left
            // the tensor pipe idle for ~400 cycles per tile: profiles/r1_spec256_trace.txt.)
            const uint64_t bd0 = make_desc_ns(smem_u32(sm.b3_tile), 128, (H / 8) * 128);
            auto issue_l3 = [&](int64_t it) {                               // D3[128,16] = A3 (TMEM) x B3^T
                const uint32_t g3 = gt + (uint32_t)it, buf3 = g3 & 1u, use3 = g3 >> 1;
                mbar_wait(&sm.a3_ready[buf3], use3 & 1u);
                tc_fence_after();
                TR(8);
                if (elect_one()) {
                    const uint32_t base = tmem_base + buf3 * 256u;
#pragma unroll
                    for (int k = 0; k < H / UMMA_K; ++k)                     // 8 TMEM columns and 256 B of B3 per K=16 step
                        umma_ts(base + C_D3, base + (uint32_t)(k * 8), bd0 + (uint64_t)(k * 16), k != 0 ? 1u : 0u);
                    umma_commit(&sm.l3_done[buf3]);
                }
                __syncwarp();
            };
            for (int64_t it = 0; it < ntiles; ++it) {
                const uint32_t g = gt + (uint32_t)it, buf = g & 1u, use = g >> 1;
                mbar_wait(&sm.d_empty[buf], (use & 1u) ^ 1u);              // E3 has read the D3 that lived in this buffer
                tc_fence_after();
                TR(0);
                const uint32_t d = tmem_base + buf * 256u;
                for (int kb = 0; kb < NKB; ++kb) {
                    if (kb == L3_SLOT && it > 0) issue_l3(it - 1);
                    mbar_wait(&sm.a_full[kb], g & 1u);
                    tc_fence_after();
                    if (kb == 0) TR(1);
                    if (kb == NKB - 1) TR(2);
                    if (elect_one()) {
                        const uint64_t ad = make_desc(smem_u32(&sm.a_tile[kb][0]));
                        const uint64_t bd = make_desc(smem_u32(&sm.b_tile[kb][0]));
#pragma unroll
                        for (int k = 0; k < KBLK / UMMA_K; ++k)              // +32 B per K=16 step inside the swizzle atom
                            umma(d, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), (kb | k) != 0 ? 1u : 0u);
                        umma_commit(&sm.a_empty[kb]);                        // slot free once these MMAs retire
                        if (kb == NKB - 1) umma_commit(&sm.d_full[buf]);     // accumulator complete
                    }
                    __syncwarp();
                }
            }
            if (ntiles > 0) issue_l3(ntiles - 1);
        } else {
            // =========================== WALKER (idle in q-table mode) ==========================
            if (!QTAB && lane == 0) {
                int iv = 2;                                                   // inventory 0
                uint64_t* codes = a.codes + (int64_t)ind * T;
                for (int64_t it = 0; it < ntiles; ++it) {
                    const uint32_t g = gt + (uint32_t)it, buf = g & 1u, use = g >> 1;
                    mbar_wait(&sm.t_full[buf], use & 1u);
                    TR(11);
                    const int64_t t0 = it * TILE_BARS;
                    const int n = (int)(T - t0 < TILE_BARS ? T - t0 : TILE_BARS);
                    const uint8_t* nb = sm.tab_n[buf];
                    if (n == TILE_BARS && !a.act_trace) walk_tile<true>(nb, sm.tab_c[buf], n, iv, codes + t0);      // every tile but the last
                    else {
                        int w = iv;
                        walk_tile<false>(nb, sm.tab_c[buf], n, iv, codes + t0);
                        if (a.act_trace) {                                    // audit: the offsets taken (second pass over the automaton)
                            for (int s = 0; s < n; ++s) {
                                int32_t* at = a.act_trace + ((int64_t)ind * T + t0 + s) * 2;
                                at[0] = sm.tab_k[buf][s * 5 + w][0]; at[1] = sm.tab_k[buf][s * 5 + w][1];
                                w = nb[s * 8 + w] & 7;
                            }
                        }
                    }
                    TR(12);
                    mbar_arrive(&sm.t_empty[buf]);
                }
            }
            __syncwarp();
        }
        tc_fence_before();
        __syncthreads();                            // every role is done with this individual's weights
        tc_fence_after();
#ifdef SGMM_SPEC256_TRACE
        if (blockIdx.x == 0 && gt == 0 && tid == 0 && ntiles >= 72) {
            const long long t00 = sm.trace[0][0];
            for (int i = 0; i < 8; ++i) {
                printf("tile %d:", 64 + i);
                for (int e = 0; e < 15; ++e) printf(" e%d=%lld", e, sm.trace[i][e] - t00);
                printf("\n");
            }
        }
#endif
        gt += (uint32_t)ntiles;
    }

    if (warp == WARP_MMA) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// one persistent CTA per SM, at most one per individual
template <bool FEE, bool QTAB>
int launch_kernel(const sgmm_bundle* b, const Args& a, cudaStream_t st)
{
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, b->device);
    const int grid = (int)(a.mm.count < sms ? a.mm.count : sms);
    const size_t smem = sizeof(Smem) + 1024;
    static std::atomic<uint64_t> configured{0};       // per instantiation, one bit per device
    if (int rc = opt_in_smem(spec256_kernel<FEE, QTAB>, smem, configured, "cudaFuncSetAttribute(spec256 smem)")) return rc;
    spec256_kernel<FEE, QTAB><<<grid, NUM_THREADS, smem, st>>>(a);
    return check_cuda(cudaGetLastError(), "spec256_kernel launch");
}

}  // namespace s256

int launch_spec256(const sgmm_bundle* b, const PopArgs& mm, double phi, double fee, double* fitness, int32_t* trades,
                   float* raw_table, int32_t* act_trace, cudaStream_t st)
{
    using namespace s256;
    if (mm.count == 0) return SGMM_OK;
    Args a{};
    a.sig = b->sig; a.px = b->px; a.T = b->T; a.tick = b->tick; a.phi = phi; a.fee = fee;
    a.mm = mm; a.fitness = fitness; a.trades = trades; a.raw_table = raw_table; a.act_trace = act_trace;
    if (int rc = reserve_codes(b, mm.count, st, &a.codes)) return rc;
    CodesRelease release(b, st);
    if (int rc = fee != 0.0 ? launch_kernel<true, false>(b, a, st) : launch_kernel<false, false>(b, a, st)) return rc;
    if (int rc = launch_account(b, a.codes, mm.count, phi, fee, fitness, trades, st)) return rc;   // the fp64 half, after the tensor-core kernel
    return release.done();
}

// With the adversary: batches of (spec256_kernel<false, true> -> q table [n][T][5], 40 B per individual and bar, in the
// bundle's code buffer under the budget of batch_bytes(); walk_account_kernel<Walk20> over it).  Seeded children need no
// staging: the kernel regenerates them.  Audit: raw_table comes from the same kernel, act_trace (the market maker's offsets
// before the displacement) from a replay of the walk over the table (launch_adv_offsets).
int launch_spec256_adv(const sgmm_bundle* b, const PopArgs& mm, const PopArgs& adv, double phi, double fee, double* fitness,
                       int32_t* trades, float* raw_table, int32_t* act_trace, cudaStream_t st)
{
    using namespace s256;
    const int64_t T = b->T;
    if (mm.count == 0) return SGMM_OK;
    int64_t nb = 0;
    uint64_t* buf = nullptr;
    if (int rc = reserve_batches(b, mm.count, 5 * T, st, &nb, &buf)) return rc;
    CodesRelease release(b, st);
    float2* q = reinterpret_cast<float2*>(buf);
    Args a{};
    a.sig = b->sig; a.px = b->px; a.T = T; a.tick = b->tick; a.phi = phi; a.fee = fee; a.qtab = q;
    const int rc = walk_batches(b, mm, &adv, nb, q, nullptr, phi, fee, fitness, trades, st,
                                [&](const PopArgs& pm, const PopArgs* pa, int64_t b0) {
        a.mm = pm;
        a.raw_table = raw_table ? raw_table + b0 * T * 10 : nullptr;
        if (int rc = launch_kernel<false, true>(b, a, st)) return rc;      // FEE is not read by the kernel body
        return act_trace ? launch_adv_offsets(b, pm.count, q, *pa, act_trace + b0 * T * 2, st) : SGMM_OK;
    });
    if (rc) return rc;
    return release.done();
}

}  // namespace sgmm
