// sgmm_tc32.cu -- H = 32 population rollout with ALL THREE policy layers on the tcgen05 tensor cores.
//
// The sequential rollout (Env/drl_engine.py:31-61) is a chain of per-individual 32x32 GEMVs.  The
// inventory is a 5-valued integer (Env/market_env.py:14-15,34-35), so the action at bar t depends on
// (t, inv) only (SURVEY.md 7.3): evaluate the policy for ALL five inventories of every bar and each
// layer becomes a GEMM whose M dimension is (bar, inventory):
//     tile = 25 bars x 5 inventories = 125 rows (+3 idle) = one M=128 tcgen05.mma
//     L1  D1[128,32] = A1[128,16] * B1^T      A1 = bf16 split of [z1, z2, inv/2, 1] (shared by the WHOLE
//                                             population: precomputed once per bundle, TMA'd to smem)
//                                             B1 = matching bf16 split of W1 | b1 (fp32-grade layer 1)
//     L2  D2[128,32] = A2[128,48] * B2^T      A2 = relu(D1) as bf16 IN TENSOR MEMORY (tcgen05.st; the MMA
//                                             reads its A operand from TMEM) | 1 | 1;  B2 = W2 | b2 hi | b2 lo
//     L3  D3[128,16] = A3[128,48] * B3^T      A3 = relu(D2) bf16 in TMEM | 1 | 1;  B3 rows 0,1 = W3 | b3 (hi),
//                                             rows 2,3 = bf16 residual of W3 | b3 (lo), rest 0
// so the CUDA cores never touch a weight: per row they only do TMEM -> cvt.rn.relu.bf16x2 -> TMEM twice,
// then quantise (x5, round-half-even, drl_engine.py:39) and take the SPECULATIVE env step of the row's
// (bar, inventory) (market_env.py:30-58) -> (fp64 reward, next inventory).  A walker lane per individual then follows
// the 5-state automaton through the table (reference order fp64 reward sum).
//
// With the ADVERSARY (drl_engine.py:42-48) the displacement depends on (fill_sell_prev, fill_buy_prev, inventory): a
// 20-state automaton.  E3 then does only the INTEGER half of the row's step for each of the four (fill_sell_prev,
// fill_buy_prev) combinations (fills against the integer thresholds, next state), the walker follows the automaton and
// MARKS the byte it visited in every bar, and the fp64 half is done for the visited rows only -- one (bar, individual)
// pair per thread of the E3 warps, with the P&L legs from a per-bar table of the reference's exact fp64 legs
// (tc32_legs_kernel, built once per (bundle, fee)) -- before the walker sums the rewards in bar order.
// Measured (profiles/r2_tc32_v*_bench.log, 4096 x 14 400): the walker must stay tiny -- it is ONE warp on a scheduler it
// shares with six busy conversion warps: doing the fp64 half of the visited rows in the walker (40 instructions per bar)
// ran at 19 ms, the marks scheme at 4.9 ms without / 6.3 ms with the adversary, leg-table rewards for every row in E3
// at 3.8 / 16.5 ms, leg records staged per chunk into a shared-memory ring by TMA (two shared loads + two fp64 adds per
// row, literal expression under a warp vote outside the record) at 3.6 ms, against 2.4 ms for the plain path below -- which
// therefore stays as it was in round 1.  The common cause: with less fp64 in E3 the MMA stream gets denser and the
// walker's 25 dependent fp64 adds per chunk -- the one piece of fp64 that cannot leave the kernel without 8 B of HBM traffic
// per env-step -- starve behind it (an fp64 instruction waits for a gap in tcgen05.mma activity, profiles/r1_fp64_under_mma.txt);
// with NO fp64 at all the kernel runs at 2.30 ms (profiles/r2_tc32_dbg1.log, dbg=1), i.e. fp64 costs 5 %, not the factor
// the shared-pipe counter suggests.  For the adversary a fifth design -- rewards of all four (fill_sell_prev, fill_buy_prev)
// combinations in E3 from a shared-memory leg ring, groups of 8 individuals with the tables in the unused operand space --
// ran at 8.5 ms at config 3's 2048 pairs against 3.25 ms for the marks scheme (profiles/r2_tc32_adv_tables_in_e3.log).  The
// adversary path is correct (tests/test_gpu_tc32.py) but not faster than the exact kernel (6.3 vs 5.3 ms): without its
// accounting it still takes 4.9 ms, with one combination instead of four 4.3 ms (profiles/r2_tc32_dbg2.log) -- the extra
// walker -> E3 -> walker round trip per chunk stalls the D3 drain, i.e. the MMA pipeline.
//
// One persistent CTA per SM works on a GROUP of up to 16 individuals in lockstep over time: the A1 tile
// of a 25-bar chunk is loaded once and multiplied with every individual's weights (a grouped GEMM:
// per-individual B operands, shared A operand), 16 walker lanes advance 16 independent automata.
//   warps 0-11  E12: three sets of four warps (warp % 4 = TMEM lane quarter), set s owns TMEM buffer s: for each
//                    of its units D1 -> relu -> bf16 -> A2 (in place), then D2 -> relu -> bf16 -> A3 (in place)
//   warps 12-23 E3 : D3 -> offsets -> speculative env step -> table; three sets of four warps, set s owns
//                    TMEM buffer s (the fp64 step is a long dependency chain: latency, not issue slots)
//   warps 24-26 L1 / L2 / L3 issuers: a converged warp each, one elected lane issues tcgen05.mma + commit
//               (three independent issue streams; the L1 warp also feeds the A1 ring with TMA bulk copies)
//   warp  27    walker
// Every TMEM region is double-buffered; per layer and buffer one "ready" mbarrier (A written + D drained)
// and one "done" mbarrier (tcgen05.commit).
//
// Precision: A2/A3/W2/W3 are bf16 (fp32 accumulate); layer 1 and all biases carry a hi+lo bf16 split.
// tests/test_gpu_tc32.py states the tolerance against the fp32 oracle and checks that GIVEN the offsets
// the kernel took, fills / inventory / trades / rewards / fitness are bit-identical to the oracle.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "sgmm_internal.h"
#include "sgmm_rng.cuh"
#include "sgmm_adversary.cuh"
#include "sgmm_step_core.h"

namespace sgmm {

namespace tc32 {

constexpr int H = 32;
constexpr int TILE_ROWS = 128;
constexpr int TILE_BARS = 25;
constexpr int GMAX = 16;                       // individuals per CTA group (even: tiles travel in pairs)
constexpr int K1 = 16, K2 = 48;
constexpr int A1_BYTES = TILE_ROWS * K1 * 2;   // 4096
constexpr int B1_BYTES = H * K1 * 2;           // 1024
constexpr int K2T = 40;                        // tf32 mode: 32 hidden + one K=8 bias step
constexpr int B2_BYTES = H * K2T * 4;          // 5120  (bf16 mode uses the first H * K2 * 2 = 3072 bytes)
constexpr int B3_BYTES = 16 * K2T * 4;         // 2560  (bf16 mode: 1536)
constexpr int A1_STAGES = 4;
constexpr int WARP_E3 = 12, WARP_L1 = 24, WARP_L2 = 25, WARP_L3 = 26;     // warp 27 = walker
constexpr int NUM_THREADS = 896;
constexpr uint32_t TMEM_COLS = 512;
// TMEM column map.  The pipeline moves UNITS of two tiles (the same 25-bar chunk for two individuals of the
// group), so that every mbarrier round trip and every issuer iteration is shared by two tiles.  Three unit
// buffers of 160 columns; inside a buffer tile j of the unit sits at + j * S_*:
//   R1 (64 columns)  D1 fp32 [128 x 32] per tile, overwritten IN PLACE by A2 = relu(D1) as bf16 pairs (16 columns)
//   R2 (64 columns)  D2 fp32, overwritten in place by A3
//   R3 (32 columns)  D3 fp32 [128 x 16] per tile
// plus 8 constant columns [1 1 0 ... 0] (bf16 pairs): the A operand of every bias K-step.
constexpr uint32_t NBUF = 3, BUF_COLS = 160;
constexpr uint32_t C_R1 = 0, C_R2 = 64, C_R3 = 128, C_ONE = 480;
constexpr uint32_t S_D = 32, S_D3 = 16;
constexpr int64_t G32 = 1250;
// operand precision of layers 2 and 3 (layer 1 is always the bf16 split): template parameter of the kernel
constexpr int M_BF16 = 0, M_TF32 = 1, M_F16 = 2;
constexpr int TAB_R_STRIDE = TILE_ROWS + 1;    // 8-byte entries per individual: 258 words -> walker lanes hit distinct banks
constexpr int TAB_N_STRIDE = 520;              // bytes per individual (25 bars x 8 B without, x 20 B with the adversary):
                                               // 130 words -> the 16 walker lanes hit distinct bank pairs
constexpr int LEG_N = 16;                      // leg table entries per bar and side: offsets K, K-1, .., K-15 (K = fill threshold)

// per-bar record of the walker's fp64 accounting: the fill thresholds and the reference's exact P&L legs
// (market_env.py:30-31,46-48,52-54) for the LEG_N offsets at and below each threshold
struct __align__(16) BarLegs {
    int32_t ka1, kb1, pad0, pad1;
    double leg_s[LEG_N];                       // (my_ask - mid_next) - my_ask*fee   at off_a = Ka - j
    double leg_b[LEG_N];                       // (mid_next - my_bid) - my_bid*fee   at off_b = Kb - j
};

struct Smem {
    uint8_t a1[A1_STAGES][A1_BYTES];
    uint8_t b1[GMAX][B1_BYTES];
    uint8_t b2[GMAX][B2_BYTES];
    uint8_t b3[GMAX][B3_BYTES];
    int2 tab_k[3][GMAX][TAB_R_STRIDE];         // quantised offsets (ka, kb) of (bar, inventory) rows; chunk q lives in buffer q % 3
    uint8_t tab_n[3][GMAX][TAB_N_STRIDE];      // next inventory index | fill_buy << 3 | fill_sell << 4: without the adversary
                                               // 8 bytes per bar (byte = entry inventory), with it 20 bytes per bar (byte = state)
    uint32_t adv_tab[GMAX][4];                 // the adversary's 20-entry displacement table of every individual (3 words)
    int2 tab_th[3][TILE_BARS + 1];             // fill thresholds + 1 (ka1, kb1) of the chunk's bars, written by E3 next to the tables
    uint64_t a1_full[A1_STAGES], a1_empty[A1_STAGES];
    // per TMEM buffer.  l*_done = tcgen05.commit of the layer's MMAs: its accumulator is complete AND the A
    // operand it read (which lives where the previous layer's accumulator was) may be overwritten.
    // a2_ready = E1 wrote A2 (4 warps); l3_ready = E2 wrote A3 (4) + E3 drained the previous D3 (4).
    uint64_t l1_done[3], a2_ready[3], l2_done[3], l3_ready[3], l3_done[3];
    uint64_t tab_full[3], tab_empty[3];
    uint64_t vis_full[3], rew_full[3];         // walker marked the visited bytes of the chunk; E3 warps wrote its rewards
    uint32_t tmem_base;
    uint32_t pad;
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
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
#ifdef SGMM_TC32_WATCHDOG
// debug build: a wait that does not complete within ~1 s reports who waits on what and traps
__device__ __noinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    const long long t0 = clock64();
    for (;;) {
        uint32_t ok;
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (ok) return;
        if (clock64() - t0 > 2000000000ll) {
            if ((threadIdx.x & 31) == 0)
                printf("tc32 watchdog: block %d warp %d waits on barrier +%u parity %u\n", (int)blockIdx.x, (int)(threadIdx.x >> 5),
                       smem_u32(bar) & 0xFFFFu, parity);
            __trap();
        }
    }
}
#else
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
#endif
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major SWIZZLE_NONE shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start>>4 | [16,30) LBO>>4 = distance between the two 16-byte k-chunks of one K=16 step
//   | [32,46) SBO>>4 = distance between 8-row groups | [46,48) version = 1 | [61,64) layout = 0
// (checked on the device by tools/tc32_unit.cu)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo)
{
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// canonical offset of element (r, k) of a [rows][K] bf16 K-major tile: 8 x 16-byte core matrices,
// k-chunks 128 B apart, 8-row groups (K/8)*128 B apart
__host__ __device__ __forceinline__ uint32_t canon(int r, int k, int K) { return (uint32_t)(((r >> 3) * (K >> 3) + (k >> 3)) * 128 + (r & 7) * 16 + (k & 7) * 2); }

// the same for 32-bit (tf32) elements: a 16-byte core-matrix row holds 4 of them
__host__ __device__ __forceinline__ uint32_t canon32(int r, int k, int K) { return (uint32_t)(((r >> 3) * (K >> 2) + (k >> 2)) * 128 + (r & 7) * 16 + (k & 3) * 4); }

// instruction descriptor: c = f32 (bit 4), a = b = bf16 (bits 7, 10), K-major both, N>>3 at [17,23), M>>4 at [24,29)
// general form: c format (0 = f16, 1 = f32) at [4,6), a / b format (0 = f16, 1 = bf16, 2 = tf32) at [7,10) / [10,13)
__host__ __device__ constexpr uint32_t idesc_any(int N, uint32_t cfmt, uint32_t afmt, uint32_t bfmt)
{
    return (cfmt << 4) | (afmt << 7) | (bfmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TILE_ROWS >> 4) << 24);
}
// tf32 operands: format code 2 at bits [7,10) and [10,13)
__host__ __device__ constexpr uint32_t idesc_tf32(int N) { return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TILE_ROWS >> 4) << 24); }
__host__ __device__ constexpr uint32_t idesc(int N) { return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TILE_ROWS >> 4) << 24); }

__device__ __forceinline__ void umma_ss(uint32_t d, uint64_t ad, uint64_t bd, uint32_t id, uint32_t acc)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
                 ::"r"(d), "l"(ad), "l"(bd), "r"(id), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_ts(uint32_t d, uint32_t a_tmem, uint64_t bd, uint32_t id, uint32_t acc)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}\n"
                 ::"r"(d), "r"(a_tmem), "l"(bd), "r"(id), "r"(acc) : "memory");
}
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
// 32 columns of 16-bit accumulators (one f16 per column) -> 16 registers of f16x2 pairs (column 2c low, 2c+1 high)
__device__ __forceinline__ void tmem_ld32_pack16(uint32_t taddr, uint32_t (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.pack::16b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ uint32_t relu_f16x2(uint32_t x)
{
    uint32_t r;
    // relu(x * 1 + (-0)) == relu(x): HFMA2.RELU runs on the FMA pipe, which this kernel leaves idle, instead of the
    // ALU pipe (HMNMX2) that the conversion and env warps compete for
    asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(x), "r"(0x3C003C00u), "r"(0x80008000u));
    return r;
}
__device__ __forceinline__ uint16_t f16_bits(float x) { return __half_as_ushort(__float2half_rn(x)); }
__device__ __forceinline__ float f16_round(float x) { return __half2float(__float2half_rn(x)); }
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
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
          "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]),
          "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]),
          "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31]) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// two fp32 -> packed bf16x2 with ReLU; `lo` lands in the low half (even k)
__device__ __forceinline__ uint32_t pack_relu_bf16(float lo, float hi)
{
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// fp32 -> tf32 (10-bit mantissa, round to nearest even), returned as fp32 bits with the low 13 bits clear
__device__ __forceinline__ uint32_t tf32_bits(float x)
{
    uint32_t r;
    asm("cvt.rn.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ uint32_t tf32_relu_bits(float x)
{
    uint32_t r;
    asm("cvt.rn.relu.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
__device__ __forceinline__ uint16_t bf16_bits(float x) { return __bfloat16_as_ushort(__float2bfloat16_rn(x)); }
// x = hi + mid + lo with each piece exactly representable in bf16 (or f16)
template <bool F16 = false>
__device__ __forceinline__ void split3(float x, float& hi, float& mid, float& lo)
{
    hi = F16 ? f16_round(x) : bf16_round(x);
    const float r1 = __fadd_rn(x, -hi);
    mid = F16 ? f16_round(r1) : bf16_round(r1);
    const float r2 = __fadd_rn(r1, -mid);
    lo = F16 ? f16_round(r2) : bf16_round(r2);
}

struct Args {
    const BarSig* sig; const BarPx* px; const uint8_t* a1; int64_t T;
    double tick, phi, fee;
    PopArgs mm, adv;
    const BarLegs* legs;     // [T] (tc32_legs_kernel)
    int32_t group;           // individuals per CTA group (<= GMAX)
    double* fitness; int32_t* trades;
    float* raw_table;        // optional audit output [P][T][5][2]
    int32_t* act_trace;      // optional audit output [P][T][2] : actions actually taken
};

// ---------------------------------------------------------------------------------------------
// bundle prologue: the layer-1 A operand of every 25-bar chunk, in the canonical K-major layout
//   k: 0 z1h 1 z1m 2 z1l 3 z1h 4 z1m 5 z1h | 6 z2h 7 z2m 8 z2l 9 z2h 10 z2m 11 z2h | 12 inv/2 13 inv/2 | 14 1 15 1
// against B1 (stage_weights): w0h w0h w0h w0m w0m w0l | w1h w1h w1h w1m w1m w1l | w2h w2m | b1h b1m
// ---------------------------------------------------------------------------------------------
// F16 = true writes the same slots as f16 pieces (the operand type of the f16 mode, whose accumulators are f16)
template <bool F16>
__global__ void tc32_a1_kernel(int64_t T, int64_t nchunks, const BarSig* __restrict__ sig, uint8_t* __restrict__ a1)
{
    auto bits = [](float x) { return F16 ? f16_bits(x) : bf16_bits(x); };
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nchunks * TILE_ROWS) return;
    const int64_t c = idx / TILE_ROWS;
    const int r = (int)(idx % TILE_ROWS);
    const int64_t t = c * TILE_BARS + r / 5;
    uint16_t v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = 0;
    if (r < TILE_BARS * 5 && t < T) {
        const float z1 = sig[t].z1, z2 = sig[t].z2;
        float h, m, l;
        split3<F16>(z1, h, m, l);
        v[0] = v[3] = v[5] = bits(h); v[1] = v[4] = bits(m); v[2] = bits(l);
        split3<F16>(z2, h, m, l);
        v[6] = v[9] = v[11] = bits(h); v[7] = v[10] = bits(m); v[8] = bits(l);
        v[12] = v[13] = bits((float)(r % 5 - 2) * 0.5f);                 // drl_engine.py:35
        v[14] = v[15] = bits(1.0f);
    }
    uint8_t* tile = a1 + c * A1_BYTES;
#pragma unroll
    for (int kc = 0; kc < 2; ++kc) {
        uint4 o;
        o.x = v[kc * 8 + 0] | ((uint32_t)v[kc * 8 + 1] << 16); o.y = v[kc * 8 + 2] | ((uint32_t)v[kc * 8 + 3] << 16);
        o.z = v[kc * 8 + 4] | ((uint32_t)v[kc * 8 + 5] << 16); o.w = v[kc * 8 + 6] | ((uint32_t)v[kc * 8 + 7] << 16);
        *reinterpret_cast<uint4*>(tile + canon(r, kc * 8, K1)) = o;
    }
}

// one genome element -> its slots in the B operands of individual slot g.  B1 (layer 1) is always the bf16
// split; B2 / B3 are bf16 (K padded to 48) or tf32 (K padded to 40).
template <int MODE>
__device__ __forceinline__ void scatter_weight(Smem& sm, int g, int e, float v)
{
    auto put = [](uint8_t* base, uint32_t off, float x) { *reinterpret_cast<uint16_t*>(base + off) = MODE == M_F16 ? f16_bits(x) : bf16_bits(x); };
    auto put32 = [](uint8_t* base, uint32_t off, uint32_t bits) { *reinterpret_cast<uint32_t*>(base + off) = bits; };
    if (e < 96) {                                      // W1[j, i]   (models/model.py:10)
        const int j = e / 3, i = e % 3;
        float h, m, l; split3<MODE == M_F16>(v, h, m, l);
        uint8_t* b = sm.b1[g];
        if (i < 2) {
            const int k0 = i * 6;
            put(b, canon(j, k0 + 0, K1), h); put(b, canon(j, k0 + 1, K1), h); put(b, canon(j, k0 + 2, K1), h);
            put(b, canon(j, k0 + 3, K1), m); put(b, canon(j, k0 + 4, K1), m); put(b, canon(j, k0 + 5, K1), l);
        } else {
            put(b, canon(j, 12, K1), h); put(b, canon(j, 13, K1), m);
        }
    } else if (e < 128) {                              // b1[j]
        const int j = e - 96;
        const float h = MODE == M_F16 ? f16_round(v) : bf16_round(v);
        const float m = __fadd_rn(v, -h);                          // rounded to the operand type by put()
        put(sm.b1[g], canon(j, 14, K1), h); put(sm.b1[g], canon(j, 15, K1), m);
    } else if (MODE == M_F16) {
        // f16 operands in the bf16 tile geometry (K padded to 48): hi = f16(v), lo = f16(v - hi) for biases and W3
        auto put16 = [](uint8_t* base, uint32_t off, uint16_t bits) { *reinterpret_cast<uint16_t*>(base + off) = bits; };
        const float hf = f16_round(v);
        const uint16_t hb = f16_bits(v), lb = f16_bits(__fadd_rn(v, -hf));
        if (e < 1152) { put16(sm.b2[g], canon((e - 128) >> 5, (e - 128) & 31, K2), hb); }
        else if (e < 1184) { put16(sm.b2[g], canon(e - 1152, 32, K2), hb); put16(sm.b2[g], canon(e - 1152, 33, K2), lb); }
        else if (e < 1248) { const int o = (e - 1184) >> 5, k = (e - 1184) & 31; put16(sm.b3[g], canon(o, k, K2), hb); put16(sm.b3[g], canon(o + 2, k, K2), lb); }
        else { const int o = e - 1248; put16(sm.b3[g], canon(o, 32, K2), hb); put16(sm.b3[g], canon(o, 33, K2), lb); }
    } else if (MODE == M_TF32) {
        // hi = tf32(v), lo = tf32(v - hi): biases and W3 carry both, W2 only hi
        const uint32_t hb = tf32_bits(v), lb = tf32_bits(__fadd_rn(v, -__uint_as_float(hb)));
        if (e < 1152) { put32(sm.b2[g], canon32((e - 128) >> 5, (e - 128) & 31, K2T), hb); }
        else if (e < 1184) { put32(sm.b2[g], canon32(e - 1152, 32, K2T), hb); put32(sm.b2[g], canon32(e - 1152, 33, K2T), lb); }
        else if (e < 1248) { const int o = (e - 1184) >> 5, k = (e - 1184) & 31; put32(sm.b3[g], canon32(o, k, K2T), hb); put32(sm.b3[g], canon32(o + 2, k, K2T), lb); }
        else { const int o = e - 1248; put32(sm.b3[g], canon32(o, 32, K2T), hb); put32(sm.b3[g], canon32(o, 33, K2T), lb); }
    } else if (e < 1152) {                             // W2[j, k]
        const int j = (e - 128) >> 5, k = (e - 128) & 31;
        put(sm.b2[g], canon(j, k, K2), v);
    } else if (e < 1184) {                             // b2[j] -> K slots 32 (hi), 33 (lo), multiplied by the constant 1 columns of A2
        const int j = e - 1152;
        const float h = bf16_round(v), m = bf16_round(__fadd_rn(v, -h));
        put(sm.b2[g], canon(j, 32, K2), h); put(sm.b2[g], canon(j, 33, K2), m);
    } else if (e < 1248) {                             // W3[o, k]: row o = hi, row o+2 = bf16 residual
        const int o = (e - 1184) >> 5, k = (e - 1184) & 31;
        const float h = bf16_round(v), m = bf16_round(__fadd_rn(v, -h));
        put(sm.b3[g], canon(o, k, K2), h); put(sm.b3[g], canon(o + 2, k, K2), m);
    } else {                                           // b3[o]
        const int o = e - 1248;
        const float h = bf16_round(v), m = bf16_round(__fadd_rn(v, -h));
        put(sm.b3[g], canon(o, 32, K2), h); put(sm.b3[g], canon(o, 33, K2), m);
    }
}

// one lane of a converged warp (the tcgen05 issue pattern: the branch is warp-uniform for the compiler)
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}\n" : "=r"(pred));
    return pred != 0;
}

// np.round(q).astype(int) (drl_engine.py:39): round-half-even.  For |q| < 2^22 the fp32 add of 1.5 * 2^23 rounds
// exactly like cvt.rni and leaves the integer in the low mantissa bits (no trip through the conversion pipe);
// larger magnitudes take the conversion instruction (saturating).
__device__ __forceinline__ int quantise(float q)
{
    if (fabsf(q) < 4194304.0f) return __float_as_int(__fadd_rn(q, 12582912.0f)) - 0x4B400000;
    return __float2int_rn(q);
}
// exact int32 -> fp64 without the conversion pipe: 2^52 + 2^31 + (k ^ 0x80000000) as a bit pattern, minus the bias
__device__ __forceinline__ double int_to_double(int k)
{
    return __dadd_rn(__hiloint2double(0x43300000, k ^ (int)0x80000000), -4503601774854144.0);
}

// The P&L leg of one filled side, the slow way: computed from the quote for an offset outside the bar's leg table (more
// than LEG_N - 1 ticks inside the fill threshold, or an always-filling bar).
__device__ __noinline__ double slow_leg(bool sell, const BarPx* px, int k, double tick, double fee)
{
    const double best = sell ? px->ask : px->bid, mid = px->mid_next;
    if (sell) return sell_leg(quote_ask(best, int_to_double(k), tick), mid, fee);
    return buy_leg(quote_bid(best, int_to_double(k), tick), mid, fee);
}

// One 25-bar chunk of one individual's walk through the table.
//   phase A: the 5-state automaton alone (a 2-instruction integer chain per bar), remembering the inventory
//            each bar was entered with;
//   phase B: rewards of the visited rows, summed in the reference's order (drl_engine.py:54); their loads do
//            not depend on the running sum, so only the fp64 add chain is serial.
// FULL = all 25 bars present (no per-bar predicates).
template <bool FULL>
__device__ __forceinline__ void walk_chunk_plain(const uint8_t* nb, const double* rb, int n, int& iv, int& trades, double& total)
{
    uint32_t es[TILE_BARS], ivs[TILE_BARS];
    uint32_t w = (uint32_t)iv;
#pragma unroll
    for (int s = 0; s < TILE_BARS; ++s) {
        ivs[s] = w; es[s] = 0;
        if (FULL || s < n) {
            const uint2 x = *reinterpret_cast<const uint2*>(nb + s * 8);
            es[s] = __byte_perm(x.x, x.y, w);          // byte `w` of the bar's 8-byte record: next | traded << 3
            w = es[s] & 7u;
        }
    }
    iv = (int)w;
#pragma unroll
    for (int s = 0; s < TILE_BARS; ++s) {
        if (FULL || s < n) {
            trades += (int)(es[s] & 8u);                                          // drl_engine.py:60-61 (x8; divided out by the caller)
            total = add_rn(total, rb[s * 5 + ivs[s]]);
        }
    }
}

// Phase A of one 25-bar chunk of one individual's walk: the automaton alone (a short integer chain per bar: 5 states,
// or 20 with the adversary).  The byte visited in every bar is marked (bit 7) for the accounting threads, trades are
// counted here (drl_engine.py:60-61).  FULL = all 25 bars present.  `st` = inventory index (0..4), with the adversary
// the state index fill_sell_prev*10 + fill_buy_prev*5 + inventory index.
template <bool ADV, bool FULL>
__device__ __forceinline__ void walk_chunk(uint8_t* nb, int n, int& st, int& trades)
{
    uint32_t cur = (uint32_t)st;
    int tr = 0;
#pragma unroll
    for (int s = 0; s < TILE_BARS; ++s) {
        if (FULL || s < n) {
            uint32_t e;
            if (!ADV) {
                const uint2 x = *reinterpret_cast<const uint2*>(nb + s * 8);
                e = __byte_perm(x.x, x.y, cur);        // byte `cur` of the bar's 8-byte record
                nb[s * 8 + cur] = (uint8_t)(e | 0x80u);
                cur = e & 7u;
            } else {
                // with the adversary the byte holds the NEXT STATE itself (5 bits) | fill_buy << 5 | fill_sell << 6: one byte
                // load at a data-dependent address per bar (latency, not instructions: the walker is short of issue slots)
                e = nb[s * 20 + cur];
                nb[s * 20 + cur] = (uint8_t)(e | 0x80u);
                cur = e & 31u;
            }
            tr += (e & (ADV ? 0x60u : 0x18u)) ? 1 : 0;
        }
    }
    st = (int)cur;
    trades += tr;
}

// position of a unit in the pipeline: TMEM buffer (unit index mod 3) and mbarrier phase parity (use count & 1)
struct Slot {
    uint32_t b, par, col;            // buffer, parity, TMEM column offset of the buffer (b * BUF_COLS)
    __device__ __forceinline__ void init(uint32_t i) { b = i % NBUF; par = (i / NBUF) & 1u; col = b * BUF_COLS; }
    template <uint32_t N>
    __device__ __forceinline__ void advance()                                                    // N <= 2 * NBUF
    {
        b += N; col += N * BUF_COLS;
        if (b >= NBUF) { b -= NBUF; col -= NBUF * BUF_COLS; par ^= 1u; }
        if (N > NBUF) { if (b >= NBUF) { b -= NBUF; col -= NBUF * BUF_COLS; par ^= 1u; } }
    }
};

// 64-bit tcgen05 operand words from 32-bit halves (the low word carries the 14-bit start address >> 4)
__device__ __forceinline__ void umma_ts2(uint32_t d, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t id, uint32_t acc)
{
    asm volatile("{\n.reg .pred p;\n.reg .b64 bd;\nsetp.ne.b32 p, %5, 0;\nmov.b64 bd, {%2, %3};\n"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], bd, %4, p;\n}\n"
                 ::"r"(d), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(id), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_ts2_tf32(uint32_t d, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t id, uint32_t acc)
{
    asm volatile("{\n.reg .pred p;\n.reg .b64 bd;\nsetp.ne.b32 p, %5, 0;\nmov.b64 bd, {%2, %3};\n"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], bd, %4, p;\n}\n"
                 ::"r"(d), "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(id), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_ss2(uint32_t d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t id, uint32_t acc)
{
    asm volatile("{\n.reg .pred p;\n.reg .b64 ad, bd;\nsetp.ne.b32 p, %6, 0;\nmov.b64 ad, {%1, %2};\nmov.b64 bd, {%3, %4};\n"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], ad, bd, %5, p;\n}\n"
                 ::"r"(d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(id), "r"(acc) : "memory");
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo) { return ((saddr >> 4) & 0x3FFFu) | (((lbo >> 4) & 0x3FFFu) << 16); }
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo) { return ((sbo >> 4) & 0x3FFFu) | (1u << 14); }     // version 1 at bit 46

// ---------------------------------------------------------------------------------------------
// The warp roles.  Each is its own (non-inlined) function so that it gets its own register allocation and
// loop optimisation; everything a role needs travels in one context record.
// ---------------------------------------------------------------------------------------------
struct Ctx {
    Smem* sm; uint32_t sm_addr;          // generic and shared-window address of the CTA's Smem
    uint32_t tmem_base, lane_addr;       // TMEM base; base + this warp's lane quarter
    uint32_t gt, gc;                     // units / chunks this CTA has processed before this group (phase sources)
    uint32_t nchunks, UG, nunits;        // this group: chunks, units per chunk, units
    uint32_t nunits_p;                   // units rounded up to a multiple of NBUF (the pad units compute on stale operands and
                                         // publish nothing): unit i of a group always lives in TMEM buffer i % NBUF, so the
                                         // buffer is a compile-time constant of the unrolled issuer loops
    int G, lane, quarter;
    int64_t grp, T, count;
    const BarSig* sig; const BarPx* px; const uint8_t* a1; const BarLegs* legs;
    double tick, phi, fee;
    double* fitness; int32_t* trades; float* raw_table; int32_t* act_trace;
};

#define BAR(member, idx) (cx.sm_addr + (uint32_t)offsetof(Smem, member) + (uint32_t)(idx) * 8u)

__device__ __forceinline__ void mbar_wait_a_(const Ctx& cx, uint32_t addr, uint32_t parity)
{
#ifdef SGMM_TC32_WATCHDOG
    // debug build: a wait that spins ~2^26 times reports who waits on what and traps
    for (uint32_t spins = 0;; ++spins) {
        uint32_t ok;
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
        if (ok) return;
        if (spins > (1u << 22)) {
            if ((threadIdx.x & 31) == 0)
                printf("tc32 watchdog: block %d warp %d waits on barrier +0x%x parity %u\n", (int)blockIdx.x, (int)(threadIdx.x >> 5), addr - BAR(a1_full, 0), parity);
            __trap();
        }
    }
#else
    // (a plain loop around one try_wait; the form with a label and a branch inside the asm statement hung the
    //  FEE instantiation of the kernel on the device although its SASS looked equivalent)
    for (;;) {
        uint32_t ok;
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
        if (ok) return;
    }
#endif
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t addr)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void umma_commit_a(uint32_t addr)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(addr) : "memory");
}

// L2 / L3 issuer: a converged warp; one elected lane issues the six MMAs of a unit and one commit
template <int LAYER, int MODE>
__device__ __noinline__ void issue_role(const Ctx& cx)
{
    constexpr bool TF32 = MODE == M_TF32;
    // layer 2 of the f16 mode accumulates in f16 (half the TMEM read traffic of the conversion); layer 3 always in fp32
    constexpr uint32_t ID = MODE == M_TF32 ? (LAYER == 2 ? idesc_tf32(32) : idesc_tf32(16))
                          : MODE == M_F16 ? (LAYER == 2 ? idesc_any(32, 0, 0, 0) : idesc_any(16, 1, 0, 0))
                                          : (LAYER == 2 ? idesc(32) : idesc(16));
    constexpr uint32_t DSTEP = LAYER == 2 ? S_D : S_D3;
    constexpr uint32_t BSTEP = (uint32_t)((LAYER == 2 ? B2_BYTES : B3_BYTES) >> 4);
    constexpr uint32_t SBO = TF32 ? (K2T / 4) * 128 : (K2 / 8) * 128;           // distance between 8-row groups of the B tile
    constexpr int KSTEPS = TF32 ? 4 : 2;                                         // data K-steps (K = 8 tf32 / 16 bf16 each)
    const uint32_t ready0 = LAYER == 2 ? BAR(a2_ready, 0) : BAR(l3_ready, 0);     // A operand written (L3: and previous D3 drained)
    const uint32_t done0 = LAYER == 2 ? BAR(l2_done, 0) : BAR(l3_done, 0);
    const uint32_t l3done0 = BAR(l3_done, 0);
    const uint32_t d0 = cx.tmem_base + (LAYER == 2 ? C_R2 : C_R3), a0 = cx.tmem_base + (LAYER == 2 ? C_R1 : C_R2);
    const uint32_t one = cx.tmem_base + C_ONE;
    const uint32_t blo0 = desc_lo(cx.sm_addr + (uint32_t)(LAYER == 2 ? offsetof(Smem, b2) : offsetof(Smem, b3)), 128), bhi = desc_hi(SBO);
    const uint32_t UG = cx.UG, nunits_p = cx.nunits_p;
    uint32_t u = 0, blo = blo0;
    uint32_t par = (cx.gt / NBUF) & 1u;                                    // cx.gt is a multiple of NBUF
#pragma unroll 1
    for (uint32_t it = 0; it < nunits_p; it += NBUF, par ^= 1u) {
#pragma unroll
        for (uint32_t bi = 0; bi < NBUF; ++bi) {                           // unit it + bi lives in buffer bi: constant offsets
            mbar_wait_a_(cx, ready0 + bi * 8u, par);
            if (LAYER == 2) mbar_wait_a_(cx, l3done0 + bi * 8u, par ^ 1u);  // layer 3 has read the A operand that lives where D2 goes
            tc_fence_after();
            if (elect_one()) {
                const uint32_t d = d0 + bi * BUF_COLS, aa = a0 + bi * BUF_COLS;
#pragma unroll
                for (int j = 0; j < 2; ++j) {                                  // the two tiles of the unit
                    const uint32_t dj = d + (uint32_t)j * DSTEP, aj = aa + (uint32_t)j * S_D, bj = blo + (uint32_t)j * BSTEP;
#pragma unroll
                    for (int k = 0; k < KSTEPS; ++k) {                         // +8 TMEM columns and +256 B of B per K-step
                        if (TF32) umma_ts2_tf32(dj, aj + 8u * k, bj + 16u * k, bhi, ID, k > 0 ? 1u : 0u);
                        else umma_ts2(dj, aj + 8u * k, bj + 16u * k, bhi, ID, k > 0 ? 1u : 0u);
                    }
                    // bias step: A = the constant [1 1 0 ...] columns
                    if (TF32) umma_ts2_tf32(dj, one, bj + 16u * KSTEPS, bhi, ID, 1u);
                    else umma_ts2(dj, one, bj + 16u * KSTEPS, bhi, ID, 1u);
                }
                umma_commit_a(done0 + bi * 8u);
            }
            __syncwarp();
            blo += 2 * BSTEP;
            if (++u == UG) { u = 0; blo = blo0; }
        }
    }
}

// L1 issuer + TMA producer of the A1 ring.  Both tiles of a unit share the A1 tile and their B1 operands are
// adjacent in shared memory (4 row groups of 256 B each): ONE M=128, N=64, K=16 MMA fills D1 of both tiles.
template <int MODE>
__device__ __noinline__ void l1_role(const Ctx& cx)
{
    const uint32_t nchunks = cx.nchunks, UG = cx.UG, nunits = cx.nunits, gc = cx.gc;
    const uint32_t a1_smem = cx.sm_addr + (uint32_t)offsetof(Smem, a1);
    auto load_a1 = [&](uint32_t c) {
        const uint32_t q = gc + c, slot = q % A1_STAGES, use = q / A1_STAGES;
        mbar_wait_a_(cx, BAR(a1_empty, slot), (use & 1u) ^ 1u);
        if (elect_one()) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(BAR(a1_full, slot)), "r"((uint32_t)A1_BYTES) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(a1_smem + slot * (uint32_t)A1_BYTES), "l"(cx.a1 + (size_t)c * A1_BYTES), "r"((uint32_t)A1_BYTES), "r"(BAR(a1_full, slot)) : "memory");
        }
        __syncwarp();
    };
    for (uint32_t c = 0; c < nchunks && c < (uint32_t)(A1_STAGES - 1); ++c) load_a1(c);
    constexpr uint32_t ID64 = MODE == M_F16 ? idesc_any(64, 0, 0, 0) : idesc(64);      // f16 mode: f16 operands and accumulator
    const uint32_t b1lo0 = desc_lo(cx.sm_addr + (uint32_t)offsetof(Smem, b1), 128), dhi = desc_hi(256);
    const uint32_t l2done0 = BAR(l2_done, 0), l1done0 = BAR(l1_done, 0);
    uint32_t c1 = 0, u1 = 0, blo = b1lo0, alo = 0, slot = 0;
    uint32_t par = (cx.gt / NBUF) & 1u;
    const uint32_t nunits_p = cx.nunits_p;
#pragma unroll 1
    for (uint32_t it = 0; it < nunits_p; it += NBUF, par ^= 1u) {
#pragma unroll
        for (uint32_t bi = 0; bi < NBUF; ++bi) {
            const bool real = it + bi < nunits;                  // pad units reuse the last A1 tile and B1 pair
            if (real && u1 == 0) {
                const uint32_t q = gc + c1;
                slot = q % A1_STAGES;
                if (c1 + A1_STAGES - 1 < nchunks) load_a1(c1 + A1_STAGES - 1);
                mbar_wait_a_(cx, BAR(a1_full, slot), (q / A1_STAGES) & 1u);
                alo = desc_lo(a1_smem + slot * (uint32_t)A1_BYTES, 128);
            }
            mbar_wait_a_(cx, l2done0 + bi * 8u, par ^ 1u);        // layer 2 of the unit that used this buffer before has read its A operand
            tc_fence_after();
            const bool last = real && (u1 + 1 == UG);
            if (elect_one()) {
                umma_ss2(cx.tmem_base + C_R1 + bi * BUF_COLS, alo, dhi, blo, dhi, ID64, 0u);
                umma_commit_a(l1done0 + bi * 8u);
                if (last) umma_commit_a(BAR(a1_empty, slot));
            }
            __syncwarp();
            if (real) {
                if (last) { u1 = 0; ++c1; blo = b1lo0; } else { ++u1; blo += 2u * (uint32_t)(B1_BYTES >> 4); }
            }
        }
    }
}

// accumulator (fp32, TMEM) -> ReLU -> bf16 pairs written back IN PLACE as the next layer's A operand, both tiles
// of a unit, this warp's 32 rows
template <int MODE>
__device__ __forceinline__ void convert_unit(uint32_t addr)
{
    if (MODE == M_F16) {
        // f16 accumulators (one per column): packed read of two columns per register, ReLU on f16 pairs, stored back
        // as the f16 A operand -- no conversion instruction at all and half the TMEM read traffic
        uint32_t h0[16], h1[16];
        tmem_ld32_pack16(addr, h0);
        tmem_ld32_pack16(addr + S_D, h1);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) h0[j] = relu_f16x2(h0[j]);
        tmem_st16(addr, h0);
#pragma unroll
        for (int j = 0; j < 16; ++j) h1[j] = relu_f16x2(h1[j]);
        tmem_st16(addr + S_D, h1);
        tmem_st_wait();
        tc_fence_before();
        return;
    }
    constexpr bool TF32 = MODE == M_TF32;
    uint32_t v0[32], v1[32];
    tmem_ld32(addr, v0);
    tmem_ld32(addr + S_D, v1);                                       // second tile of the unit
    tmem_ld_wait();
    if (TF32) {                                                      // fp32 -> relu -> tf32, 32 columns back in place
#pragma unroll
        for (int j = 0; j < 32; ++j) v0[j] = tf32_relu_bits(__uint_as_float(v0[j]));
        tmem_st32(addr, v0);
#pragma unroll
        for (int j = 0; j < 32; ++j) v1[j] = tf32_relu_bits(__uint_as_float(v1[j]));
        tmem_st32(addr + S_D, v1);
    } else {                                                         // fp32 -> relu -> bf16 pairs, 16 columns
#pragma unroll
        for (int j = 0; j < 16; ++j) v0[j] = pack_relu_bf16(__uint_as_float(v0[2 * j]), __uint_as_float(v0[2 * j + 1]));
        tmem_st16(addr, reinterpret_cast<uint32_t (&)[16]>(v0));
#pragma unroll
        for (int j = 0; j < 16; ++j) v1[j] = pack_relu_bf16(__uint_as_float(v1[2 * j]), __uint_as_float(v1[2 * j + 1]));
        tmem_st16(addr + S_D, reinterpret_cast<uint32_t (&)[16]>(v1));
    }
    tmem_st_wait();
    tc_fence_before();
}

// E12: set s (four warps) owns TMEM buffer s: for each of its units it converts D1 -> A2, then D2 -> A3
template <int MODE>
__device__ __noinline__ void convert_role(const Ctx& cx, uint32_t set)
{
    const uint32_t it0 = set;                                    // cx.gt is a multiple of NBUF: unit it lives in buffer it % NBUF
    uint32_t par = (cx.gt / NBUF) & 1u;
    const uint32_t r1 = cx.lane_addr + C_R1 + set * BUF_COLS, r2 = cx.lane_addr + C_R2 + set * BUF_COLS;
    const uint32_t l1_done = BAR(l1_done, set), a2_ready = BAR(a2_ready, set), l2_done = BAR(l2_done, set), l3_ready = BAR(l3_ready, set);
    const uint32_t nunits = cx.nunits_p;                         // the pad units are converted too (keeps the barrier phases in step)
    const bool leader = cx.lane == 0;
#pragma unroll 1
    for (uint32_t it = it0; it < nunits; it += NBUF, par ^= 1u) {
        mbar_wait_a_(cx, l1_done, par);
        tc_fence_after();
        convert_unit<MODE>(r1);
        __syncwarp();
        if (leader) mbar_arrive_a(a2_ready);
        mbar_wait_a_(cx, l2_done, par);
        tc_fence_after();
        convert_unit<MODE>(r2);
        __syncwarp();
        if (leader) mbar_arrive_a(l3_ready);
    }
}

// PLAIN path (no adversary), as measured in round 1 -- E3: D3 -> offsets -> speculative env step of every (bar, inventory) row -> table.  Set s (four warps) owns TMEM
// buffer s, i.e. the units with (global unit index % 3) == s: consecutive uses of its barriers, so every parity
// wait is at most one phase away.  Outer loop over chunks (bar data, table buffer), inner loop over the set's
// units of the chunk.
template <bool FEE>
__device__ __noinline__ void e3_role_plain(const Ctx& cx, uint32_t e3set)
{
    Smem& sm = *cx.sm;
    const int lane = cx.lane;
    const int row = cx.quarter * 32 + lane;
    const int tl = row / 5, iv = row % 5;            // bar within the chunk, inventory index (inv+2)
    const bool row_ok = row < TILE_BARS * 5;
    const int64_t T = cx.T;
    const uint32_t nchunks = cx.nchunks, UG = cx.UG, gc = cx.gc, gt = cx.gt;
    const BarSig* sig = cx.sig; const BarPx* px = cx.px;
    const double tick = cx.tick, phi = cx.phi, fee = cx.fee;
    int2 kth = make_int2(0, 0), kth_n = make_int2(0, 0);
    double2 ab = make_double2(0., 0.), ab_n = make_double2(0., 0.);
    double mid = 0.0, mid_n = 0.0;
    auto load_bar = [&](uint32_t c, int2& k, double2& q, double& m) {
        const int64_t t = (int64_t)c * TILE_BARS + tl;
        if (row_ok && t < T) {
            k = __ldg(reinterpret_cast<const int2*>(&sig[t].ka1));
            q = __ldg(reinterpret_cast<const double2*>(&px[t].ask));
            m = __ldg(&px[t].mid_next);
        }
    };
    const uint32_t taddr = cx.lane_addr + C_R3 + e3set * BUF_COLS;
    const uint32_t l3_done = BAR(l3_done, e3set), l3_ready = BAR(l3_ready, e3set);
    uint32_t par = (gt / NBUF) & 1u;                                            // cx.gt is a multiple of NBUF
    uint32_t base3 = 0;                                                         // (index of the chunk's first unit) % 3
    const uint32_t ug3 = UG % NBUF;
    const int inv = iv - 2;
    const bool leader = lane == 0;
    if (nchunks > 0) load_bar(0, kth_n, ab_n, mid_n);
#pragma unroll 1
    for (uint32_t c = 0; c < nchunks; ++c) {
        kth = kth_n; ab = ab_n; mid = mid_n;
        if (c + 1 < nchunks) load_bar(c + 1, kth_n, ab_n, mid_n);               // prefetch the next chunk's bars
        uint32_t up = e3set >= base3 ? e3set - base3 : e3set + NBUF - base3;    // first unit of the chunk that is ours
        base3 += ug3; if (base3 >= NBUF) base3 -= NBUF;
        if (up >= UG) continue;                                                 // (groups of 2 or 4: not every chunk has one)
        const uint32_t q = gc + c, cbuf = q % 3u;
        const bool valid = row_ok && ((int64_t)c * TILE_BARS + tl < T);
        mbar_wait_a_(cx, BAR(tab_empty, cbuf), ((q / 3u) & 1u) ^ 1u);                // walker has left this table buffer
        const uint32_t tab_full = BAR(tab_full, cbuf);
        double* tr = reinterpret_cast<double*>(&sm.tab_k[cbuf][up * 2u][row]);
        uint8_t* tn = &sm.tab_n[cbuf][up * 2u][tl * 8 + iv];
#pragma unroll 1
        for (; up < UG; up += NBUF, par ^= 1u, tr += 2 * NBUF * TAB_R_STRIDE, tn += 2 * NBUF * TAB_N_STRIDE) {
            mbar_wait_a_(cx, l3_done, par);
            tc_fence_after();
            uint32_t v[2][4];
            tmem_ld4(taddr, v[0]);
            tmem_ld4(taddr + S_D3, v[1]);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (leader) mbar_arrive_a(l3_ready);                                 // accumulator drained
            // Both tiles of the unit, branch-free so that the two dependency chains interleave.  Rows that
            // are not valid compute on stale bar data and store nothing.
            float ra[2], rb[2]; double rew[2]; uint32_t nxt[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                ra[j] = __fadd_rn(__uint_as_float(v[j][0]), __uint_as_float(v[j][2]));       // hi + lo halves of W3
                rb[j] = __fadd_rn(__uint_as_float(v[j][1]), __uint_as_float(v[j][3]));
                const int ka = quantise(__fmul_rn(ra[j], 5.0f));                             // drl_engine.py:39
                const int kb = quantise(__fmul_rn(rb[j], 5.0f));
                // speculative env step of (bar t, inventory iv-2)  (market_env.py:30-58)
                const bool fb = (inv < 2) && (kb < kth.y);                   // :34,:37
                const bool fs = (inv > -2) && (ka < kth.x);                  // :35,:38
                const double leg_s = sell_leg<FEE>(quote_ask(ab.x, int_to_double(ka), tick), mid, fee);
                const double leg_b = buy_leg<FEE>(quote_bid(ab.y, int_to_double(kb), tick), mid, fee);
                double pnl = 0.0;
                pnl = fb ? add_rn(pnl, leg_b) : pnl;
                pnl = fs ? add_rn(pnl, leg_s) : pnl;
                const int ninv = inv + (fb ? 1 : 0) - (fs ? 1 : 0);
                const double pen = mul_rn(phi, int_to_double(ninv < 0 ? -ninv : ninv));            // phi * |inv'|  (:57)
                rew[j] = sub_rn(pnl, pen);                                                         // :58
                nxt[j] = (uint32_t)(ninv + 2) | ((fb || fs) ? 8u : 0u);
            }
            if (valid) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    tr[j * TAB_R_STRIDE] = rew[j];
                    tn[j * TAB_N_STRIDE] = (uint8_t)nxt[j];
                }
                if (cx.raw_table) {
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int64_t ind = cx.grp * cx.G + (int64_t)(up * 2u) + j;
                        if (ind < cx.count) {
                            float* o = cx.raw_table + (((int64_t)ind * T + (int64_t)c * TILE_BARS + tl) * 5 + iv) * 2;
                            __stcg(o, ra[j]); __stcg(o + 1, rb[j]);
                        }
                    }
                }
            }
            __syncwarp();
            if (leader) mbar_arrive_a(tab_full);
        }
    }
    // pad units of the group (at most two, one per set): drain the accumulator so that the barrier phases stay in step
    for (uint32_t it = cx.nunits; it < cx.nunits_p; ++it) {
        if (it % NBUF != e3set) continue;
        mbar_wait_a_(cx, l3_done, par);
        tc_fence_after();
        uint32_t v[4];
        tmem_ld4(taddr, v);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (leader) mbar_arrive_a(l3_ready);
        par ^= 1u;
    }
}

// walker: one lane per individual of the group
__device__ __noinline__ void walker_role_plain(const Ctx& cx)
{
    Smem& sm = *cx.sm;
    const int g = cx.lane;
    const int64_t ind = cx.grp * cx.G + g, T = cx.T;
    const bool live = g < cx.G && ind < cx.count;
    const uint32_t nchunks = cx.nchunks, gc = cx.gc;
    int iv = 2, trades = 0;                                       // inventory 0
    double total = 0.0;                                           // drl_engine.py:26
#pragma unroll 1
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t q = gc + c, cbuf = q % 3u, cpar = (q / 3u) & 1u;
        mbar_wait_a_(cx, BAR(tab_full, cbuf), cpar);
        if (live) {
            const int64_t t0 = (int64_t)c * TILE_BARS;
            const int n = (int)(T - t0 < TILE_BARS ? T - t0 : TILE_BARS);
            const uint8_t* nb = sm.tab_n[cbuf][g];
            const double* rb = reinterpret_cast<const double*>(sm.tab_k[cbuf][g]);
            if (n == TILE_BARS && !cx.act_trace) walk_chunk_plain<true>(nb, rb, n, iv, trades, total);      // every chunk but the last
            else {
                const int iv0 = iv;
                walk_chunk_plain<false>(nb, rb, n, iv, trades, total);
                if (cx.act_trace) {                                    // audit: the offsets taken (second pass over the automaton)
                    int w = iv0;
                    for (int s = 0; s < n; ++s) {
                        const float* o = cx.raw_table + (((int64_t)ind * T + t0 + s) * 5 + w) * 2;
                        int32_t* at = cx.act_trace + ((int64_t)ind * T + t0 + s) * 2;
                        at[0] = quantise(__fmul_rn(__ldcg(o), 5.0f));
                        at[1] = quantise(__fmul_rn(__ldcg(o + 1), 5.0f));
                        w = nb[s * 8 + w] & 7;
                    }
                }
            }
        }
        __syncwarp();
        if (cx.lane == 0) mbar_arrive_a(BAR(tab_empty, cbuf));
    }
    if (live) {
        trades >>= 3;                                                  // walk_chunk_plain counts in units of 8
        cx.fitness[ind] = episode_fitness(total, trades); cx.trades[ind] = trades;
    }
}

// The fp64 half of the env step for the rows the walker visited in chunk c, one (bar, individual) pair per thread of
// the twelve E3 warps: find the marked byte of the pair's bar record (-> the state the bar was entered with, fills, next
// inventory), the offsets of that row, the adversary's displacement, the legs of the sides that filled from the bar's
// leg table (market_env.py:30-31,44-55) and reward = pnl - phi*|inventory| (:57-58), stored as a double over the bar's
// first row of the offset table (dead by now) for the walker's bar-order sum.
template <bool ADV>
__device__ __forceinline__ void account_chunk(const Ctx& cx, uint32_t c, const PenaltyTable& pen)
{
    Smem& sm = *cx.sm;
    const uint32_t q = cx.gc + c, cbuf = q % 3u;
    mbar_wait_a_(cx, BAR(vis_full, cbuf), (q / 3u) & 1u);
    const int64_t t0 = (int64_t)c * TILE_BARS;
    const int n = (int)(cx.T - t0 < TILE_BARS ? cx.T - t0 : TILE_BARS);
    const int a = ((int)(threadIdx.x >> 5) - WARP_E3) * 32 + cx.lane;
    const int npairs = cx.G * TILE_BARS;
    for (int p = a; p < npairs; p += 12 * 32) {
        const int g = p / TILE_BARS, s = p - g * TILE_BARS;
        const int64_t ind = cx.grp * cx.G + g;
        if (s >= n || ind >= cx.count) continue;
        uint32_t idx, e;
        if (!ADV) {
            const uint2 x = *reinterpret_cast<const uint2*>(&sm.tab_n[cbuf][g][s * 8]);
            const uint32_t m0 = x.x & 0x80808080u;
            idx = m0 ? (uint32_t)(__ffs((int)m0) - 1) >> 3 : 4u;
            e = __byte_perm(x.x, x.y, idx) & 0x7Fu;
        } else {
            const uint32_t* x = reinterpret_cast<const uint32_t*>(&sm.tab_n[cbuf][g][s * 20]);
            uint32_t w = 0, wi = 0;
#pragma unroll
            for (int i = 4; i >= 0; --i) { const uint32_t v = x[i]; if (v & 0x80808080u) { w = v; wi = (uint32_t)i; } }
            const uint32_t b = (uint32_t)(__ffs((int)(w & 0x80808080u)) - 1) >> 3;
            idx = wi * 4u + b;
            e = (w >> (8u * b)) & 0x7Fu;
        }
        const bool fb = (e & (ADV ? 32u : 8u)) != 0, fs = (e & (ADV ? 64u : 16u)) != 0;
        const int iv_in = ADV ? (int)(idx % 5u) : (int)idx;
        const int niv = ADV ? (int)((e & 31u) % 5u) : (int)(e & 7u);
        int2 k = sm.tab_k[cbuf][g][s * 5 + iv_in];
        if (cx.act_trace) { int32_t* at = cx.act_trace + ((int64_t)ind * cx.T + t0 + s) * 2; at[0] = k.x; at[1] = k.y; }   // audit: the offsets taken
        if (ADV) {
            const uint32_t d = table_lookup(sm.adv_tab[g][0], sm.adv_tab[g][1], sm.adv_tab[g][2], (int)idx);
            k.x += (int)(d & 3u) - 1; k.y += (int)(d >> 2) - 1;                      // market_env.py:26-28
        }
        const int2 th = sm.tab_th[cbuf][s];
        const BarLegs* L = cx.legs + t0 + s;
        double lb = 0.0, ls = 0.0;
        if (fb) {                                                                      // :44-49
            const long long j = (long long)th.y - 1 - k.y;
            lb = (unsigned long long)j < (unsigned long long)LEG_N ? __ldg(&L->leg_b[j]) : slow_leg(false, cx.px + t0 + s, k.y, cx.tick, cx.fee);
        }
        if (fs) {                                                                      // :50-55
            const long long j = (long long)th.x - 1 - k.x;
            ls = (unsigned long long)j < (unsigned long long)LEG_N ? __ldg(&L->leg_s[j]) : slow_leg(true, cx.px + t0 + s, k.x, cx.tick, cx.fee);
        }
        // pnl = 0.0 (+ leg_b) (+ leg_s) in the reference's order (:40,:48,:54); 0.0 + leg == leg (a leg is never -0.0)
        const double pnl = fb ? (fs ? add_rn(lb, ls) : lb) : ls;
        *reinterpret_cast<double*>(&sm.tab_k[cbuf][g][s * 5]) = sub_rn(pnl, penalty(pen, abs(niv - 2)));      // :58
    }
    __syncwarp();
    if (cx.lane == 0) mbar_arrive_a(BAR(rew_full, cbuf));
}

// E3: D3 -> offsets -> the INTEGER half of the speculative env step of every (bar, inventory) row -> tables.  Set s
// (four warps) owns TMEM buffer s, i.e. the units with (global unit index % 3) == s: consecutive uses of its barriers,
// so every parity wait is at most one phase away.  Outer loop over chunks (bar thresholds, table buffer), inner loop
// over the set's units of the chunk.  With the adversary the row's fills are decided for each of the four
// (fill_sell_prev, fill_buy_prev) combinations (drl_engine.py:42-48: the displacement depends on them and on the inventory).
template <bool ADV>
__device__ __noinline__ void e3_role(const Ctx& cx, uint32_t e3set)
{
    Smem& sm = *cx.sm;
    const int lane = cx.lane;
    const int row = cx.quarter * 32 + lane;
    const int tl = row / 5, iv = row % 5;            // bar within the chunk, inventory index (inv+2)
    const bool row_ok = row < TILE_BARS * 5;
    const int64_t T = cx.T;
    const uint32_t nchunks = cx.nchunks, UG = cx.UG, gc = cx.gc, gt = cx.gt;
    const BarSig* sig = cx.sig;
    int2 kth = make_int2(0, 0), kth_n = make_int2(0, 0);
    auto load_bar = [&](uint32_t c, int2& k) {
        const int64_t t = (int64_t)c * TILE_BARS + tl;
        if (row_ok && t < T) k = __ldg(reinterpret_cast<const int2*>(&sig[t].ka1));
    };
    const uint32_t taddr = cx.lane_addr + C_R3 + e3set * BUF_COLS;
    const uint32_t l3_done = BAR(l3_done, e3set), l3_ready = BAR(l3_ready, e3set);
    uint32_t par = (gt / NBUF) & 1u;                                            // cx.gt is a multiple of NBUF
    uint32_t base3 = 0;                                                         // (index of the chunk's first unit) % 3
    const uint32_t ug3 = UG % NBUF;
    const int inv = iv - 2;
    const bool leader = lane == 0;
    const bool can_buy = inv < 2, can_sell = inv > -2;                          // market_env.py:34-35
    const PenaltyTable pen = penalty_table(cx.phi);
    if (nchunks > 0) load_bar(0, kth_n);
#pragma unroll 1
    for (uint32_t c = 0; c < nchunks; ++c) {
        kth = kth_n;
        if (c + 1 < nchunks) load_bar(c + 1, kth_n);                            // prefetch the next chunk's thresholds
        uint32_t up = e3set >= base3 ? e3set - base3 : e3set + NBUF - base3;    // first unit of the chunk that is ours
        base3 += ug3; if (base3 >= NBUF) base3 -= NBUF;
        if (up >= UG) { if (c >= 1) account_chunk<ADV>(cx, c - 1, pen); continue; }     // (groups of 2 or 4: not every chunk has a unit of ours)
        const uint32_t q = gc + c, cbuf = q % 3u;
        const bool valid = row_ok && ((int64_t)c * TILE_BARS + tl < T);
        mbar_wait_a_(cx, BAR(tab_empty, cbuf), ((q / 3u) & 1u) ^ 1u);                // walker has left this table buffer
        const uint32_t tab_full = BAR(tab_full, cbuf);
        if (row_ok && iv == 0) sm.tab_th[cbuf][tl] = kth;                       // every set writes the same values: benign
        int2* tk = &sm.tab_k[cbuf][up * 2u][row];
        uint8_t* tn = &sm.tab_n[cbuf][up * 2u][ADV ? tl * 20 + iv : tl * 8 + iv];
        const uint32_t* advt = &sm.adv_tab[up * 2u][0];
#pragma unroll 1
        for (; up < UG; up += NBUF, par ^= 1u, tk += 2 * NBUF * TAB_R_STRIDE, tn += 2 * NBUF * TAB_N_STRIDE, advt += 2 * NBUF * 4) {
            mbar_wait_a_(cx, l3_done, par);
            tc_fence_after();
            uint32_t v[2][4];
            tmem_ld4(taddr, v[0]);
            tmem_ld4(taddr + S_D3, v[1]);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (leader) mbar_arrive_a(l3_ready);                                 // accumulator drained
            // Both tiles of the unit, branch-free.  Rows that are not valid compute on stale thresholds and store nothing.
            float ra[2], rb[2]; int ka[2], kb[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                ra[j] = __fadd_rn(__uint_as_float(v[j][0]), __uint_as_float(v[j][2]));       // hi + lo halves of W3
                rb[j] = __fadd_rn(__uint_as_float(v[j][1]), __uint_as_float(v[j][3]));
                ka[j] = max(min(quantise(__fmul_rn(ra[j], 5.0f)), K_CLAMP), -K_CLAMP);        // drl_engine.py:39
                kb[j] = max(min(quantise(__fmul_rn(rb[j], 5.0f)), K_CLAMP), -K_CLAMP);
            }
            if (!ADV) {
                uint32_t e[2];
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const bool fb = can_buy && (kb[j] < kth.y);                  // market_env.py:34,37
                    const bool fs = can_sell && (ka[j] < kth.x);                 // :35,:38
                    e[j] = (uint32_t)(iv + (fb ? 1 : 0) - (fs ? 1 : 0)) | (fb ? 8u : 0u) | (fs ? 16u : 0u);      // :45,:51
                }
                if (valid) {
#pragma unroll
                    for (int j = 0; j < 2; ++j) { tk[j * TAB_R_STRIDE] = make_int2(ka[j], kb[j]); tn[j * TAB_N_STRIDE] = (uint8_t)e[j]; }
                }
            } else {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const uint4 at = *reinterpret_cast<const uint4*>(advt + j * 4);
                    uint32_t e[4];
#pragma unroll
                    for (int cmb = 0; cmb < 4; ++cmb) {                          // cmb = fill_sell_prev*2 + fill_buy_prev
                        const uint32_t d = table_lookup(at.x, at.y, at.z, cmb * 5 + iv);
                        const int oa = ka[j] + (int)(d & 3u) - 1, ob = kb[j] + (int)(d >> 2) - 1;    // :26-28
                        const bool fb = can_buy && (ob < kth.y);
                        const bool fs = can_sell && (oa < kth.x);
                        e[cmb] = (uint32_t)((fs ? 10 : 0) + (fb ? 5 : 0) + iv + (fb ? 1 : 0) - (fs ? 1 : 0)) | (fb ? 32u : 0u) | (fs ? 64u : 0u);
                    }
                    if (valid) {
                        tk[j * TAB_R_STRIDE] = make_int2(ka[j], kb[j]);
#pragma unroll
                        for (int cmb = 0; cmb < 4; ++cmb) tn[j * TAB_N_STRIDE + cmb * 5] = (uint8_t)e[cmb];
                    }
                }
            }
            if (valid && cx.raw_table) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int64_t ind = cx.grp * cx.G + (int64_t)(up * 2u) + j;
                    if (ind < cx.count) {
                        float* o = cx.raw_table + (((int64_t)ind * T + (int64_t)c * TILE_BARS + tl) * 5 + iv) * 2;
                        __stcg(o, ra[j]); __stcg(o + 1, rb[j]);
                    }
                }
            }
            __syncwarp();
            if (leader) mbar_arrive_a(tab_full);
        }
        // the fp64 half of the PREVIOUS chunk's visited rows (the walker has marked them by now), all E3 warps
        if (c >= 1) account_chunk<ADV>(cx, c - 1, pen);
    }
    if (nchunks >= 1) account_chunk<ADV>(cx, nchunks - 1, pen);
    // pad units of the group (at most two, one per set): drain the accumulator so that the barrier phases stay in step
    for (uint32_t it = cx.nunits; it < cx.nunits_p; ++it) {
        if (it % NBUF != e3set) continue;
        mbar_wait_a_(cx, l3_done, par);
        tc_fence_after();
        uint32_t v[4];
        tmem_ld4(taddr, v);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (leader) mbar_arrive_a(l3_ready);
        par ^= 1u;
    }
}

// walker: one lane per individual of the group.  Per chunk: the automaton (phase A, marks the visited bytes), then --
// one chunk behind, when the E3 warps have turned the marks into rewards -- the reference-order fp64 sum.
template <bool ADV>
__device__ __noinline__ void walker_role(const Ctx& cx)
{
    Smem& sm = *cx.sm;
    const int g = cx.lane;
    const int64_t ind = cx.grp * cx.G + g, T = cx.T;
    const bool live = g < cx.G && ind < cx.count;
    const uint32_t nchunks = cx.nchunks, gc = cx.gc;
    int st = 2, trades = 0;                                       // inventory 0, no previous fills
    double total = 0.0;                                           // drl_engine.py:26
    auto sum_chunk = [&](uint32_t c) {
        const uint32_t q = gc + c, cbuf = q % 3u;
        mbar_wait_a_(cx, BAR(rew_full, cbuf), (q / 3u) & 1u);
        if (live) {
            const int64_t t0 = (int64_t)c * TILE_BARS;
            const int n = (int)(T - t0 < TILE_BARS ? T - t0 : TILE_BARS);
            const double* rw = reinterpret_cast<const double*>(&sm.tab_k[cbuf][g][0]);
            if (n == TILE_BARS) {
#pragma unroll
                for (int s = 0; s < TILE_BARS; ++s) total = add_rn(total, rw[s * 5]);          // drl_engine.py:54
            } else {
                for (int s = 0; s < n; ++s) total = add_rn(total, rw[s * 5]);
            }
        }
        __syncwarp();
        if (cx.lane == 0) mbar_arrive_a(BAR(tab_empty, cbuf));
    };
#pragma unroll 1
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t q = gc + c, cbuf = q % 3u, cpar = (q / 3u) & 1u;
        {   // pull the next chunk's leg records (25 x 272 B) into L1 for the accounting threads
            const int64_t tn0 = (int64_t)(c + 1) * TILE_BARS;
            if (tn0 < T) {
                const int64_t nb_ = T - tn0 < TILE_BARS ? T - tn0 : TILE_BARS;
                const char* p0 = reinterpret_cast<const char*>(cx.legs + tn0);
                for (int64_t off = (int64_t)cx.lane * 128; off < nb_ * (int64_t)sizeof(BarLegs); off += 32 * 128)
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(p0 + off));
            }
        }
        mbar_wait_a_(cx, BAR(tab_full, cbuf), cpar);
        if (live) {
            const int64_t t0 = (int64_t)c * TILE_BARS;
            const int n = (int)(T - t0 < TILE_BARS ? T - t0 : TILE_BARS);
            uint8_t* nb = sm.tab_n[cbuf][g];
            if (n == TILE_BARS) walk_chunk<ADV, true>(nb, n, st, trades);          // every chunk but the last
            else walk_chunk<ADV, false>(nb, n, st, trades);
        }
        __syncwarp();
        if (cx.lane == 0) mbar_arrive_a(BAR(vis_full, cbuf));
        if (c >= 1) sum_chunk(c - 1);
    }
    if (nchunks >= 1) sum_chunk(nchunks - 1);
    if (live) { cx.fitness[ind] = episode_fitness(total, trades); cx.trades[ind] = trades; }
}

template <bool ADV, bool FEE, int MODE>
__global__ void __launch_bounds__(NUM_THREADS, 1) tc32_kernel(const Args a)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t misalign = smem_u32(smem_raw) & 127u;
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw + ((128u - misalign) & 127u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t T = a.T;
    const int G = a.group;
    const uint32_t nchunks = (uint32_t)((T + TILE_BARS - 1) / TILE_BARS);
    const uint32_t UG = (uint32_t)G >> 1;                       // units (pairs of individuals) per chunk
    const uint32_t nunits = nchunks * UG;

    if (tid == 0) {
        for (int i = 0; i < A1_STAGES; ++i) { mbar_init(&sm.a1_full[i], 1); mbar_init(&sm.a1_empty[i], 1); }
        for (int i = 0; i < NBUF; ++i) {
            mbar_init(&sm.l1_done[i], 1); mbar_init(&sm.a2_ready[i], 4);
            mbar_init(&sm.l2_done[i], 1); mbar_init(&sm.l3_ready[i], 8); mbar_init(&sm.l3_done[i], 1);
        }
        for (int i = 0; i < 3; ++i) {
            mbar_init(&sm.tab_full[i], 4u * UG); mbar_init(&sm.tab_empty[i], 1);
            mbar_init(&sm.vis_full[i], 1); mbar_init(&sm.rew_full[i], 12);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == WARP_L1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // B operands: the padding (K slots 34..47, B3 rows 4..15) stays zero for the whole kernel
    for (int i = tid; i < GMAX * (B1_BYTES + B2_BYTES + B3_BYTES) / 16; i += NUM_THREADS)
        reinterpret_cast<uint4*>(&sm.b1[0][0])[i] = make_uint4(0, 0, 0, 0);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sm.tmem_base;
    const int quarter = warp & 3;                    // TMEM lane quarter this warp may touch (warp % 4)
    const uint32_t e3set = (uint32_t)(warp - WARP_E3) >> 2;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    if (warp < 4) {
        // the constant K-step shared by every layer-2 / layer-3 MMA: K slots 32, 33 = 1.0 (they meet the
        // bias rows of B2 / B3), 34..47 = 0
        constexpr bool TF32 = MODE == M_TF32;
        uint32_t c[8] = {TF32 ? 0x3F800000u : (MODE == M_F16 ? 0x3C003C00u : 0x3F803F80u), TF32 ? 0x3F800000u : 0u, 0, 0, 0, 0, 0, 0};
        tmem_st8(lane_addr + C_ONE, c);
        tmem_st_wait();
    }
    // "previous accumulator drained" half of the first use of the l3_ready barriers
    if (warp >= WARP_E3 && warp < WARP_L1 && lane == 0) mbar_arrive(&sm.l3_ready[e3set]);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const PopArgs pop = resolve(a.mm);
    const PopArgs advpop = ADV ? resolve(a.adv) : a.adv;
    Ctx cx;
    cx.sm = &sm; cx.sm_addr = smem_u32(&sm); cx.tmem_base = tmem_base; cx.lane_addr = lane_addr;
    cx.gt = 0; cx.gc = 0; cx.nchunks = nchunks; cx.UG = UG; cx.nunits = nunits;
    cx.nunits_p = (nunits + NBUF - 1) / NBUF * NBUF;
    cx.G = G; cx.lane = lane; cx.quarter = quarter; cx.T = T; cx.count = pop.count;
    cx.sig = a.sig; cx.px = a.px; cx.a1 = a.a1; cx.legs = a.legs; cx.tick = a.tick; cx.phi = a.phi; cx.fee = a.fee;
    cx.fitness = a.fitness; cx.trades = a.trades; cx.raw_table = a.raw_table; cx.act_trace = a.act_trace;

    for (int64_t grp = blockIdx.x; grp * G < pop.count; grp += gridDim.x) {
        // ---------------- stage the group's weights (all warps) ----------------------------------
        for (int task = tid; task < G * 313; task += NUM_THREADS) {
            const int g = task / 313, q = task % 313;
            const int64_t ind = grp * G + g;
            const bool live = ind < pop.count;
            const GenomeSource src = make_source(pop, live ? ind : 0, G32);
            const int e0 = q * 4;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (live) {
                if (q < 312) src.at4(e0, v);
                else { v[0] = src.at(e0); v[1] = src.at(e0 + 1); }
            }
            if (MODE == M_BF16 && e0 >= 128 && e0 < 1152) {     // 4 consecutive k of one W2 row: one 8-byte store
                const int j = (e0 - 128) >> 5, k = (e0 - 128) & 31;
                uint2 o;
                o.x = bf16_bits(v[0]) | ((uint32_t)bf16_bits(v[1]) << 16);
                o.y = bf16_bits(v[2]) | ((uint32_t)bf16_bits(v[3]) << 16);
                *reinterpret_cast<uint2*>(sm.b2[g] + canon(j, k, K2)) = o;
            } else {
                const int n = q < 312 ? 4 : 2;
                for (int i = 0; i < n; ++i) scatter_weight<MODE>(sm, g, e0 + i, v[i]);
            }
        }
        if (ADV) {
            // the adversary of every individual of the group as its 20-entry displacement table (sgmm_adversary.cuh)
            if (tid < GMAX * 4) (&sm.adv_tab[0][0])[tid] = 0u;
            __syncthreads();
            for (int task = tid; task < G * 20; task += NUM_THREADS) {
                const int g = task / 20, st = task % 20;
                const int64_t ind = grp * G + g;
                uint32_t e = 5u;                                       // (0, 0)
                if (ind < pop.count) e = adversary_entry(make_source(advpop, ind, G32), st);
                atomicOr(&sm.adv_tab[g][st >> 3], e << ((st & 7) * 4));
            }
        }
        fence_proxy_async();                       // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncthreads();

        cx.grp = grp;
        if (warp < WARP_E3) convert_role<MODE>(cx, (uint32_t)warp >> 2);
        else if (warp < WARP_L1) { if (ADV) e3_role<true>(cx, e3set); else e3_role_plain<FEE>(cx, e3set); }
        else if (warp == WARP_L1) l1_role<MODE>(cx);
        else if (warp == WARP_L2) issue_role<2, MODE>(cx);
        else if (warp == WARP_L3) issue_role<3, MODE>(cx);
        else if (ADV) walker_role<true>(cx);
        else walker_role_plain(cx);

        cx.gt += cx.nunits_p;
        cx.gc += nchunks;
        tc_fence_before();
        __syncthreads();                            // every role is done with this group's weights and tables
        tc_fence_after();
    }

    if (warp == WARP_L1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

}  // namespace tc32

int tc32_chunks(int64_t T) { return (int)((T + tc32::TILE_BARS - 1) / tc32::TILE_BARS); }
size_t tc32_a1_bytes(int64_t T) { return 2 * (size_t)tc32_chunks(T) * tc32::A1_BYTES; }   // bf16 tiles, then f16 tiles

int launch_tc32_prologue(sgmm_bundle* b, cudaStream_t st)
{
    using namespace tc32;
    if (b->T == 0) return SGMM_OK;
    const int64_t nchunks = tc32_chunks(b->T);
    const int64_t n = nchunks * TILE_ROWS;
    tc32_a1_kernel<false><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(b->T, nchunks, b->sig, b->a1);
    tc32_a1_kernel<true><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(b->T, nchunks, b->sig, b->a1 + nchunks * A1_BYTES);
    return check_cuda(cudaGetLastError(), "tc32_a1_kernel launch");
}

// individuals per CTA group: minimise waves x group (the time of one launch), prefer the larger group
int tc32_group_size(int64_t count, int sms)
{
    int best = 2; int64_t best_cost = INT64_MAX;
    for (int g = 2; g <= tc32::GMAX; g += 2) {
        const int64_t groups = (count + g - 1) / g;
        const int64_t waves = (groups + sms - 1) / sms;
        const int64_t cost = waves * g;
        if (cost <= best_cost) { best_cost = cost; best = g; }
    }
    return best;
}

// The walker's per-bar records: thresholds + the reference's exact fp64 legs for the LEG_N offsets at and below each
// threshold (one thread per (bar, side, j)); fee terms always evaluated, like the reference does with fee_rate = 0.
__global__ void tc32_legs_kernel(int64_t T, const BarSig* __restrict__ sig, const BarPx* __restrict__ px, double tick, double fee,
                                 tc32::BarLegs* __restrict__ legs)
{
    using namespace tc32;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= T * 2 * LEG_N) return;
    const int64_t t = idx / (2 * LEG_N);
    const int r = (int)(idx % (2 * LEG_N)), side = r / LEG_N, j = r % LEG_N;
    const int32_t k1 = side == 0 ? sig[t].ka1 : sig[t].kb1;
    if (r == 0) { legs[t].ka1 = sig[t].ka1; legs[t].kb1 = sig[t].kb1; legs[t].pad0 = legs[t].pad1 = 0; }
    double leg = 0.0;
    if (k1 != K_NEVER && k1 != K_ALWAYS) {                          // (never-filling bars need no legs; always-filling ones take the slow path)
        const long long k = (long long)k1 - 1 - j;
        if (k >= -(long long)K_CLAMP - 1 && k <= (long long)K_CLAMP + 1) {
            const BarPx p = px[t];
            if (side == 0) leg = sell_leg(quote_ask(p.ask, int_to_double((int)k), tick), p.mid_next, fee);
            else leg = buy_leg(quote_bid(p.bid, int_to_double((int)k), tick), p.mid_next, fee);
        }
    }
    (side == 0 ? legs[t].leg_s : legs[t].leg_b)[j] = leg;
}

// leg tables of a bundle, one per fee rate seen (tick is a property of the bundle); built on first use on the caller's
// stream, later users on other streams wait for the build through an event
int tc32_legs(const sgmm_bundle* cb, double fee, cudaStream_t st, const tc32::BarLegs** out)
{
    using namespace tc32;
    sgmm_bundle* b = const_cast<sgmm_bundle*>(cb);
    *out = nullptr;
    if (b->T == 0) return SGMM_OK;                                  // an empty episode visits no bar
    std::lock_guard<std::mutex> lock(b->legs_mutex);
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (st) cudaStreamIsCapturing(st, &cap);
    for (auto& e : b->legs) {
        if (memcmp(&e.fee, &fee, sizeof fee) == 0) {
            if (e.stream != st && cap == cudaStreamCaptureStatusNone)
                if (int rc = check_cuda(cudaStreamWaitEvent(st, e.ready, 0), "cudaStreamWaitEvent(leg table)")) return rc;
            *out = reinterpret_cast<const BarLegs*>(e.buf);
            return SGMM_OK;
        }
    }
    if (cap != cudaStreamCaptureStatusNone) {
        set_error("the bundle has no leg table for fee_rate %g yet: run one tensor-core rollout with this fee outside the stream capture first", fee);
        return SGMM_ERR_INVALID;
    }
    if (b->legs.size() >= 64) { set_error("more than 64 distinct fee rates on one bundle (each keeps a %zu-byte leg table)", (size_t)b->T * sizeof(BarLegs)); return SGMM_ERR_NOMEM; }
    sgmm_bundle::LegTable e;
    e.fee = fee; e.stream = st;
    if (int rc = check_cuda(cudaMalloc(&e.buf, (size_t)b->T * sizeof(BarLegs)), "cudaMalloc(leg table)")) return rc;
    if (int rc = check_cuda(cudaEventCreateWithFlags(&e.ready, cudaEventDisableTiming), "cudaEventCreate(leg table)")) { cudaFree(e.buf); return rc; }
    const int64_t n = b->T * 2 * LEG_N;
    tc32_legs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(b->T, b->sig, b->px, b->tick, fee, reinterpret_cast<BarLegs*>(e.buf));
    int rc = check_cuda(cudaGetLastError(), "tc32_legs_kernel launch");
    if (!rc) rc = check_cuda(cudaEventRecord(e.ready, st), "cudaEventRecord(leg table)");
    if (rc) { cudaFree(e.buf); cudaEventDestroy(e.ready); return rc; }
    b->legs.push_back(e);
    *out = reinterpret_cast<const BarLegs*>(e.buf);
    return SGMM_OK;
}

int launch_tc32(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, double phi, double fee, int group, double* fitness, int32_t* trades,
                float* raw_table, int32_t* act_trace, cudaStream_t st, int mode)
{
    using namespace tc32;
    if (mm.count == 0) return SGMM_OK;
    if (act_trace && !raw_table) { set_error("act_trace needs raw_table"); return SGMM_ERR_INVALID; }
    Args a;
    a.legs = nullptr;
    if (adv) if (int rc = tc32_legs(b, fee, st, &a.legs)) return rc;     // only the adversary path accounts through the leg table
    a.sig = b->sig; a.px = b->px; a.a1 = b->a1 + (mode == M_F16 ? tc32_chunks(b->T) * A1_BYTES : 0); a.T = b->T; a.tick = b->tick; a.phi = phi; a.fee = fee;
    a.mm = mm; a.fitness = fitness; a.trades = trades; a.raw_table = raw_table; a.act_trace = act_trace;
    if (adv) a.adv = *adv; else { PopArgs z = {}; a.adv = z; }
    const int sms = sm_count(b->device);
    a.group = (group >= 2 && group <= GMAX && group % 2 == 0) ? group : tc32_group_size(mm.count, sms);
    const int64_t groups = (mm.count + a.group - 1) / a.group;
    const int grid = (int)(groups < sms ? groups : sms);
    const size_t smem = sizeof(Smem) + 128;
    static std::atomic<uint64_t> configured[9];       // per variant, one bit per device (zero-initialised)
    if (mode < 0 || mode > 2) { set_error("unknown tensor-core mode %d", mode); return SGMM_ERR_INVALID; }
    const int sub = adv ? 2 : (fee != 0.0 ? 1 : 0);            // plain, plain with fee, adversary
    const int variant = sub + 3 * mode;
    void (*kern)(const Args) = nullptr;
    switch (variant) {
        case 0: kern = tc32_kernel<false, false, M_BF16>; break;
        case 1: kern = tc32_kernel<false, true, M_BF16>; break;
        case 2: kern = tc32_kernel<true, false, M_BF16>; break;
        case 3: kern = tc32_kernel<false, false, M_TF32>; break;
        case 4: kern = tc32_kernel<false, true, M_TF32>; break;
        case 5: kern = tc32_kernel<true, false, M_TF32>; break;
        case 6: kern = tc32_kernel<false, false, M_F16>; break;
        case 7: kern = tc32_kernel<false, true, M_F16>; break;
        default: kern = tc32_kernel<true, false, M_F16>; break;
    }
    if (int rc = opt_in_smem(kern, smem, configured[variant], "cudaFuncSetAttribute(tc32 smem)")) return rc;
    kern<<<grid, NUM_THREADS, smem, st>>>(a);
    return check_cuda(cudaGetLastError(), "tc32_kernel launch");
}

}  // namespace sgmm
