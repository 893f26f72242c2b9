// sgmm_exact256.cu -- bit-exact (SGMM-F32 order) episodes at hidden width 256 (BASELINE config 4's policy width).
//
// The exact H = 32 kernels keep a whole individual's weights in registers; at H = 256 the hidden layer alone is 256 KB of
// fp32, so the episode takes the split of the small-population path (sgmm_one.cu) instead:
//   1. exact256_table_kernel  the exact policy for EVERY (bar, inventory) pair of a batch of individuals: per individual a
//                             [5T x 256] x [256 x 256] fp32 product on the CUDA cores (no tensor cores: every product and
//                             every sum must round exactly as the oracle's, oracle/sgmm_oracle.c:105-164), plus the same
//                             per-pair output as one::policy_table_kernel (step code + next inventory, or q = raw*5 for the
//                             adversary's walk, or raw itself for the trace kernel);
//   2. the walk kernels of sgmm_one.cu, unchanged (prefix scan over the inventory automaton, reference-order fp64 sum).
//
// Table kernel: one CTA = 8 warps computes BM = 32 pairs x all 256 hidden units.  Thread (warp w, lane) owns the rows
// rg, rg+8, rg+16, rg+24 (rg = lane / 4) and the columns l, l+32, ..., l+224 (l = 4w + lane % 4): the 8 columns of ONE lane
// of the oracle's layer-3 reduction, so the output layer's per-lane fma chain over b = 1..7 runs in registers and only the
// 32-lane butterfly goes through shared memory (as warp shuffles, in the oracle's xor order 16, 8, 4, 2, 1).
// Layer 2 keeps the four chains k mod 4 of every output as two float2 accumulators (chains (0,1) and (2,3): one packed
// fma.rn.f32x2 each per k-group of four); W2 streams through shared memory in K-slices of 32 in ascending k (the
// accumulation order is fixed by k, not by the slicing), double-buffered with cp.async; h1 of the tile stays in shared
// memory for the whole K.  Per k-group a warp issues 12 shared loads (4 h1 rows broadcast over the lanes that share
// them, 8 W2 columns broadcast over the 8 row groups) for 64 FFMA2.
#include <cstdio>
#include <cstdlib>
#include "sgmm_internal.h"
#include "sgmm_rng.cuh"

namespace sgmm {

namespace x256 {

constexpr int H = 256;
constexpr int64_t G = (int64_t)H * H + 7 * H + 2;     // 67 330 floats
constexpr int BM = 32;                                 // (bar, inventory) pairs per tile
constexpr int THREADS = 256;
constexpr int KS = 32;                                 // k per W2 slice
constexpr int KGS = KS / 4;                            // k-groups of four per slice
constexpr int NSLICE = H / KS;
constexpr int OFF_B1 = 3 * H, OFF_W2 = 4 * H, OFF_B2 = 4 * H + H * H, OFF_W3 = 5 * H + H * H, OFF_B3 = 7 * H + H * H;

struct Smem {
    float4 h1[H / 4][BM];           // h1[kg][row] = h1 of the row at k = 4kg .. 4kg+3               32 KB
    float4 w2[2][KGS][H];           // w2[buf][kg][j] = W2[j, k0+4kg .. k0+4kg+3]                    64 KB
    float4 l1[H];                   // {W1[j,0], W1[j,1], W1[j,2], b1[j]}                             4 KB
    float b2[H];
    float2 w3[H];                   // {W3[0,j], W3[1,j]}
    float2 part[BM][32];            // layer-3 lane sums p_l of every row (a, b)                      8 KB
    float4 in[BM];                  // z1, z2, tha, thb of the row's bar
    float b3[2];
};

__device__ __forceinline__ void cp_async8(void* dst, const void* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// W2[:, 32s .. 32s+31] of genome row g -> sm.w2[buf]: 4096 8-byte copies, 16 per thread; four consecutive threads
// read 32 contiguous bytes of one W2 row
__device__ __forceinline__ void load_slice(Smem& sm, int buf, const float* __restrict__ g, int s)
{
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int idx = threadIdx.x + THREADS * i;
        const int half = idx & 1, kg = ((idx >> 10) << 1) | ((idx >> 1) & 1), j = (idx >> 2) & 255;
        const float* src = g + OFF_W2 + (int64_t)j * H + s * KS + 4 * kg + 2 * half;
        cp_async8(reinterpret_cast<float2*>(&sm.w2[buf][kg][j]) + half, src);
    }
    cp_async_commit();
}

// Phase probe (build with SGMM_EXTRA_NVCC_FLAGS=-DSGMM_EXACT256_PROBE): lane 0 of every warp of CTA 0 sums clock64 deltas
// of the task prologue + layer 1, of the waits for each W2 slice (cp.async + barrier), of the FFMA2 loop, of the barrier
// after it, and of the epilogue, and prints them when the CTA ends.
#ifdef SGMM_EXACT256_PROBE
#define X256_MARK(acc) do { const long long now_ = clock64(); acc += now_ - probe_t; probe_t = now_; } while (0)
#else
#define X256_MARK(acc) do { } while (0)
#endif

// mode: 0 plain (step code + next inventory, one::policy_table_kernel's format), 1 q = raw*5 per pair (adversary walk),
//       2 raw per pair (trace kernel)
__global__ void __launch_bounds__(THREADS, 1) exact256_table_kernel(const BarSig* __restrict__ sig, int64_t T,
                                                                     const float* __restrict__ genomes, int64_t count, int mode,
                                                                     float2* __restrict__ code, uint8_t* __restrict__ next)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rg = lane >> 2, l = warp * 4 + (lane & 3);
    const int64_t pairs = T * 5, tiles = (pairs + BM - 1) / BM, ntasks = count * tiles;
    int64_t loaded = -1;
#ifdef SGMM_EXACT256_PROBE
    long long probe_t = clock64(), c_pro = 0, c_wait = 0, c_ffma = 0, c_bar = 0, c_epi = 0, n_tasks = 0;
#endif
    for (int64_t task = blockIdx.x; task < ntasks; task += gridDim.x) {
        const int64_t ind = task / tiles, p0 = (task - ind * tiles) * BM;
        const float* g = genomes + ind * G;
        load_slice(sm, 0, g, 0);                                   // W2 slice 0 flies while layer 1 runs
        if (ind != loaded) {                                       // small weights of the individual (the previous task is done with them)
            for (int j = tid; j < H; j += THREADS) {
                sm.l1[j] = make_float4(__ldg(g + 3 * j), __ldg(g + 3 * j + 1), __ldg(g + 3 * j + 2), __ldg(g + OFF_B1 + j));
                sm.b2[j] = __ldg(g + OFF_B2 + j);
                sm.w3[j] = make_float2(__ldg(g + OFF_W3 + j), __ldg(g + OFF_W3 + H + j));
            }
            if (tid < 2) sm.b3[tid] = __ldg(g + OFF_B3 + tid);
            loaded = ind;
        }
        if (tid < BM) {
            const int64_t p = p0 + tid < pairs ? p0 + tid : pairs - 1;
            const int64_t t = p / 5;
            const float4 s = __ldg(reinterpret_cast<const float4*>(&sig[t]));             // z1, z2, tha, thb
            sm.in[tid] = s;
        }
        __syncthreads();
        // ---- layer 1: a = b1; a = fma(W1[j,0], z1, a); fma(W1[j,1], z2, a); fma(W1[j,2], inv/2, a); ReLU ----
#pragma unroll 2
        for (int e = tid; e < BM * (H / 4); e += THREADS) {
            const int row = e & (BM - 1), kg = e / BM;
            const int64_t p = p0 + row < pairs ? p0 + row : pairs - 1;
            const float inv2 = (float)((int)(p % 5) - 2) * 0.5f;                          // drl_engine.py:35
            const float4 x = sm.in[row];
            float h[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float4 w = sm.l1[4 * kg + i];
                float v = __fmaf_rn(w.x, x.x, w.w);
                v = __fmaf_rn(w.y, x.y, v);
                v = __fmaf_rn(w.z, inv2, v);
                h[i] = fmaxf(v, 0.0f);
            }
            sm.h1[kg][row] = make_float4(h[0], h[1], h[2], h[3]);
        }
        // ---- layer 2: chains (c0, c1) and (c2, c3) of output (row, j) as two packed accumulators ----
        float2 acc01[4][8], acc23[4][8];
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const float bias = sm.b2[l + 32 * b];
#pragma unroll
            for (int r = 0; r < 4; ++r) { acc01[r][b] = make_float2(bias, 0.0f); acc23[r][b] = make_float2(0.0f, 0.0f); }
        }
#pragma unroll 1
        for (int s = 0; s < NSLICE; ++s) {
            if (s + 1 < NSLICE) { load_slice(sm, (s + 1) & 1, g, s + 1); cp_async_wait<1>(); }
            else cp_async_wait<0>();
            if (s == 0) X256_MARK(c_pro);
            __syncthreads();                                       // slice s (and, at s = 0, h1) visible to every warp
            X256_MARK(c_wait);
            const float4 (*w2)[H] = sm.w2[s & 1];
#pragma unroll
            for (int kg = 0; kg < KGS; ++kg) {
                float4 h[4];
#pragma unroll
                for (int r = 0; r < 4; ++r) h[r] = sm.h1[s * KGS + kg][rg + 8 * r];
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    const float4 w = w2[kg][l + 32 * b];
                    const float2 wlo = make_float2(w.x, w.y), whi = make_float2(w.z, w.w);
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        acc01[r][b] = __ffma2_rn(wlo, make_float2(h[r].x, h[r].y), acc01[r][b]);
                        acc23[r][b] = __ffma2_rn(whi, make_float2(h[r].z, h[r].w), acc23[r][b]);
                    }
                }
            }
            X256_MARK(c_ffma);
            __syncthreads();                                       // buffer s & 1 free for slice s + 2
            X256_MARK(c_bar);
        }
        // ---- h2 = ReLU((c0 + c2) + (c1 + c3)); layer 3 lane l: W3[o,l]*h2[l], then fma over b = 1..7 ----
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            float pa = 0.0f, pb = 0.0f;
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                const float2 S = __fadd2_rn(acc01[r][b], acc23[r][b]);                  // (c0+c2, c1+c3)
                const float h2 = fmaxf(__fadd_rn(S.x, S.y), 0.0f);
                const float2 w3 = sm.w3[l + 32 * b];
                if (b == 0) { pa = __fmul_rn(w3.x, h2); pb = __fmul_rn(w3.y, h2); }
                else { pa = __fmaf_rn(w3.x, h2, pa); pb = __fmaf_rn(w3.y, h2, pb); }
            }
            sm.part[rg + 8 * r][l] = make_float2(pa, pb);
        }
        __syncthreads();
        // ---- butterfly over the 32 lane sums (xor 16, 8, 4, 2, 1), + b3, and the pair's output: warp w, rows 4w..4w+3 ----
#pragma unroll
        for (int i = 0; i < BM / 8; ++i) {
            const int row = warp * (BM / 8) + i;
            const float2 v = sm.part[row][lane];
            float ra = v.x, rb = v.y;
#pragma unroll
            for (int m = 16; m >= 1; m >>= 1) {
                ra = __fadd_rn(ra, __shfl_xor_sync(0xffffffffu, ra, m));
                rb = __fadd_rn(rb, __shfl_xor_sync(0xffffffffu, rb, m));
            }
            const int64_t p = p0 + row;
            if (lane != 0 || p >= pairs) continue;
            ra = __fadd_rn(ra, sm.b3[0]); rb = __fadd_rn(rb, sm.b3[1]);
            float2* codei = code + ind * pairs;
            if (mode == 2) { codei[p] = make_float2(ra, rb); continue; }
            const float qa = __fmul_rn(ra, 5.0f), qb = __fmul_rn(rb, 5.0f);                 // raw*5.0 (drl_engine.py:39)
            if (mode == 1) { codei[p] = make_float2(qa, qb); continue; }
            const int64_t t = p / 5;
            const int iv = (int)(p - t * 5);
            const float inv2 = (float)(iv - 2) * 0.5f;
            const float4 s = sm.in[row];
            // integer half of the env step, rounding folded into the per-bar float thresholds (as one::policy_table_kernel)
            const bool fb = (inv2 < 1.0f) && (qb < s.w);                                     // market_env.py:34,37
            const bool fs = (inv2 > -1.0f) && (qa < s.z);                                    // :35,:38
            codei[p] = make_float2(fs ? qa : __int_as_float(SGMM_CODE_NOFILL_F), fb ? qb : __int_as_float(SGMM_CODE_NOFILL_F));
            next[ind * T * 8 + t * 8 + iv] = (uint8_t)(iv + (fb ? 1 : 0) - (fs ? 1 : 0));      // :45,:51
        }
        __syncthreads();                                           // h1, part and the row inputs are reused by the next task
        X256_MARK(c_epi);
#ifdef SGMM_EXACT256_PROBE
        ++n_tasks;
#endif
    }
#ifdef SGMM_EXACT256_PROBE
    if (blockIdx.x == 0 && lane == 0)
        printf("x256 probe warp %d tasks %lld cycles/task: prologue+layer1 %lld slice-wait %lld ffma2-loop %lld after-loop-barrier %lld epilogue %lld\n",
               warp, n_tasks, c_pro / n_tasks, c_wait / n_tasks, c_ffma / n_tasks, c_bar / n_tasks, c_epi / n_tasks);
#endif
}

// explicit genome rows (8-byte aligned copies) or seeded children, materialised once per batch: [count][G]
__global__ void __launch_bounds__(256) stage_genomes_kernel(const PopArgs mm_in, int64_t count, float* __restrict__ out)
{
    const PopArgs mm = resolve(mm_in);
    constexpr int64_t per = (G + 3) / 4;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < count * per; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t ind = idx / per, q = idx - ind * per;
        const GenomeSource src = make_source(mm, ind, G);
        float* o = out + ind * G + 4 * q;
        if (4 * q + 4 <= G) {
            float v[4]; src.at4(4 * q, v);
            o[0] = v[0]; o[1] = v[1]; o[2] = v[2]; o[3] = v[3];
        } else {
            for (int64_t e = 4 * q; e < G; ++e) out[ind * G + e] = src.at(e);
        }
    }
}

constexpr int64_t DEFAULT_BATCH_BYTES = (int64_t)2 << 30;

// bytes of scratch a batch may use: SGMM_EXACT256_BATCH_BYTES (read on every call), else 2 GiB
int64_t batch_bytes()
{
    const char* e = getenv("SGMM_EXACT256_BATCH_BYTES");
    const long long v = e ? atoll(e) : 0;
    return v > 0 ? (int64_t)v : DEFAULT_BATCH_BYTES;
}

int launch_table(const sgmm_bundle* b, const float* rows, int64_t count, int mode, float2* code, uint8_t* next, cudaStream_t st)
{
    if (b->T == 0 || count == 0) return SGMM_OK;
    static std::atomic<uint64_t> configured{0};
    if (int rc = opt_in_smem(exact256_table_kernel, sizeof(Smem), configured, "cudaFuncSetAttribute(exact256 smem)")) return rc;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, b->device);
    const int64_t tasks = count * ((b->T * 5 + BM - 1) / BM);
    const int64_t blocks = tasks < sms ? tasks : sms;
    exact256_table_kernel<<<(unsigned)blocks, THREADS, sizeof(Smem), st>>>(b->sig, b->T, rows, count, mode, code, next);
    return check_cuda(cudaGetLastError(), "exact256_table_kernel launch");
}

int launch_stage(const sgmm_bundle* b, const PopArgs& mm, int64_t count, float* out, cudaStream_t st)
{
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, b->device);
    const int64_t work = count * ((G + 3) / 4);
    const int64_t want = (work + 255) / 256, cap = (int64_t)sms * 8;
    stage_genomes_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(mm, count, out);
    return check_cuda(cudaGetLastError(), "stage_genomes_kernel launch");
}

bool needs_stage(const PopArgs& mm) { return mm.genomes == nullptr || (reinterpret_cast<uintptr_t>(mm.genomes) & 7u) != 0; }

}  // namespace x256

int reserve_batches(const sgmm_bundle* b, int64_t P, int64_t per_ind, cudaStream_t st, int64_t* nb, uint64_t** buf)
{
    const int64_t T = b->T;
    int64_t n = x256::batch_bytes() / (per_ind * 8 > 0 ? per_ind * 8 : 1);
    if (n < 1) n = 1;
    if (n > P) n = P;
    *nb = n;
    const int64_t units = T > 0 ? (n * per_ind + T - 1) / T + 1 : 1;           // reserve_codes counts in units of T words
    return reserve_codes(b, units, st, buf);
}

// Episodes at H = 256 in SGMM-F32 order (with or without the adversary): batches of individuals, each batch = (staged
// genomes,) policy table, walk.  The table ([n][T] x 48 B) and the staged genomes ([n] x 269 KB; seeded children, or
// explicit rows not 8-byte aligned) live in the bundle's grow-only code buffer (sgmm_account.cu), under the byte budget of
// x256::batch_bytes(); rollouts sharing the buffer are ordered across streams, and the first rollout of a size allocates
// and must not run under a stream capture.
int launch_exact256(const sgmm_bundle* b, const PopArgs& mm, const PopArgs* adv, double phi, double fee, double* fitness, int32_t* trades,
                    cudaStream_t st)
{
    using namespace x256;
    const int64_t T = b->T, P = mm.count;
    if (P == 0) return SGMM_OK;
    const bool stage = T > 0 && needs_stage(mm);
    int64_t nb = 0;
    uint64_t* buf = nullptr;
    if (int rc = reserve_batches(b, P, 6 * T + (stage ? G / 2 : 0), st, &nb, &buf)) return rc;
    CodesRelease release(b, st);
    float2* code = reinterpret_cast<float2*>(buf);
    uint8_t* next = reinterpret_cast<uint8_t*>(code + nb * T * 5);
    float* staged = reinterpret_cast<float*>(buf + nb * T * 6);
    const int rc = walk_batches(b, mm, adv, nb, code, next, phi, fee, fitness, trades, st, [&](const PopArgs& pm, const PopArgs*, int64_t) {
        const float* rows = pm.genomes;
        if (stage) {
            if (int rc = launch_stage(b, pm, pm.count, staged, st)) return rc;
            rows = staged;
        }
        return launch_table(b, rows, pm.count, adv ? 1 : 0, code, next, st);
    });
    if (rc) return rc;
    return release.done();
}

// raw policy outputs (before x5) of ONE explicit genome for every (bar, inventory): out = float2[T][5].  `stage_buf` holds
// G floats for a genome that is not 8-byte aligned.
int launch_exact256_raw(const sgmm_bundle* b, const float* genome, float2* out, float* stage_buf, cudaStream_t st)
{
    using namespace x256;
    PopArgs pm{};
    pm.genomes = genome; pm.count = 1;
    const float* rows = genome;
    if (needs_stage(pm)) {
        if (int rc = launch_stage(b, pm, 1, stage_buf, st)) return rc;
        rows = stage_buf;
    }
    return launch_table(b, rows, 1, 2, out, nullptr, st);
}

}  // namespace sgmm
