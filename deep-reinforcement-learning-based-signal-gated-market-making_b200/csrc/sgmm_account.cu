// sgmm_account.cu -- the fp64 half of the tensor-core rollouts, run AFTER the rollout kernel.
//
// Measured on B200 (tools/walk_bench.cu, profiles/r1_fp64_under_mma.txt): while tcgen05.mma instructions execute,
// an FP64 instruction of the same SM waits ~740 cycles instead of 9 (100 dependent DADDs: 921 cycles on an idle SM,
// 74 146 with back-to-back N=256 MMAs) -- integer, shared-memory and shuffle instructions are unaffected.  The
// reference's accounting is fp64 by definition (Env/market_env.py:30-58, Env/drl_engine.py:54), so the tensor-core
// kernels do only the INTEGER half of the env step (offsets, fills, inventory) and record, per bar actually visited,
// a 64-bit code; this kernel turns the codes into rewards (the fp64 step arithmetic of sgmm_step_core.h: quotes, legs,
// penalty, the no-trade rule) and sums them in the reference's order:
//     code = (fill_sell ? off_a : SGMM_CODE_NOFILL) | (fill_buy ? off_b : SGMM_CODE_NOFILL) << 32      (two int32)
// (an offset is only needed on a side that filled; the inventory is re-derived here as the running sum of the fills).
// The exact H=32 kernel (sgmm_rollout.cu) uses the same split INSIDE one kernel: its compute warps hand the step
// records through shared memory to the CTA's producer warp, which accounts all individuals of the CTA (lane =
// individual).  Here the codes go through global memory because the H=256 kernel works on one individual per CTA
// and its fp64 would run next to the MMAs whichever warp issued it.
#include "sgmm_internal.h"
#include "sgmm_step_core.h"

namespace sgmm {

namespace {

// A CTA accounts ACC_IND individuals.  Warp w < ACC_IND turns the codes of 32 consecutive bars of individual w into
// rewards (lane = bar; coalesced code loads; the fp64 legs only on lanes whose bar traded) and puts them into a
// shared-memory tile; the last warp is the summing warp: its lane j adds individual j's 32 rewards in bar order
// (drl_engine.py:54) -- the only serial part, 32 individuals' chains side by side in one instruction stream --
// while the other warps already work on the next 32 bars (two tiles).
constexpr int ACC_IND = 4;                                       // small CTAs: 4096 individuals spread evenly over 148 SMs
constexpr int ACC_THREADS = (ACC_IND + 1) * 32;
constexpr int ACC_STRIDE = 33;                                   // doubles per tile row: conflict-free column reads

template <bool FEE, bool FLT>
__global__ void __launch_bounds__(ACC_THREADS) account_kernel(const uint64_t* __restrict__ codes, const BarPx* __restrict__ px,
                                                              int64_t T, int64_t count, double tick, double phi, double fee,
                                                              double* __restrict__ fitness, int32_t* __restrict__ trades)
{
    __shared__ double tile[2][ACC_IND][ACC_STRIDE];
    __shared__ int s_trades[ACC_IND];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t ind0 = (int64_t)blockIdx.x * ACC_IND;
    const int64_t nwin = (T + 31) / 32;
    if (warp < ACC_IND) {
        // ---------------- rewards of individual ind0 + warp, 32 bars per window ----------------
        const int64_t ind = ind0 + warp;
        const bool live = ind < count;
        const uint64_t* c = codes + (live ? ind : 0) * T;
        int ntr = 0, inv = 0;                                        // market_env.py:17 (reset)
        const PenaltyTable pen = penalty_table(phi);
        const uint64_t none = FLT ? 0xFFFFFFFFFFFFFFFFull : 0x8000000080000000ull;            // no fills beyond T
        uint64_t code_n = (live && lane < T) ? __ldcs(c + lane) : none;                       // window 0
        // the bars' prices are loaded unconditionally one window ahead (L1/L2-resident: every individual reads the same
        // bars); loading them only on the lanes that traded put an L2 round trip on every window's critical path
        double2 ab_n = make_double2(0.0, 0.0); double mid_n = 0.0;
        if (lane < T) { ab_n = __ldg(reinterpret_cast<const double2*>(&px[lane].ask)); mid_n = __ldg(&px[lane].mid_next); }
        for (int64_t w = 0; w < nwin; ++w) {
            const int64_t t = w * 32 + lane;
            const uint64_t code = code_n;
            const int64_t tn = t + 32;
            code_n = (live && tn < T) ? __ldcs(c + tn) : none;                                   // prefetch the next window
            const double2 ab = ab_n; const double mid = mid_n;
            if (tn < T) { ab_n = __ldg(reinterpret_cast<const double2*>(&px[tn].ask)); mid_n = __ldg(&px[tn].mid_next); }
            int ka = (int)(uint32_t)code, kb = (int)(uint32_t)(code >> 32);
            const bool fs = ka != (FLT ? SGMM_CODE_NOFILL_F : SGMM_CODE_NOFILL), fb = kb != (FLT ? SGMM_CODE_NOFILL_F : SGMM_CODE_NOFILL);
            // inventory after each bar = running sum of the fills (market_env.py:45,51): two ballots instead of a scan
            const uint32_t mb = __ballot_sync(0xffffffffu, fb), ms = __ballot_sync(0xffffffffu, fs);
            const uint32_t le = 0xffffffffu >> (31 - lane);                             // lanes 0..lane
            const int ninv = inv + __popc(mb & le) - __popc(ms & le);
            inv += __popc(mb) - __popc(ms);
            const bool traded = fb || fs;
            ntr += __popc(mb | ms);                                                     // drl_engine.py:60-61
            const int ai = ninv < 0 ? -ninv : ninv;
            double pnl = 0.0;                                                           // market_env.py:40
            if (traded) {
                if (fb) {
                    if (FLT) kb = __float2int_rn(__int_as_float(kb));                   // drl_engine.py:39 (np.round, half to even)
                    pnl = add_rn(pnl, buy_leg<FEE>(quote_bid(ab.y, kb, tick), mid, fee));
                }
                if (fs) {
                    if (FLT) ka = __float2int_rn(__int_as_float(ka));
                    pnl = add_rn(pnl, sell_leg<FEE>(quote_ask(ab.x, ka, tick), mid, fee));
                }
            }
            tile[w & 1][warp][lane] = sub_rn(pnl, penalty(pen, ai));                    // market_env.py:58
            __syncthreads();                                                            // tile w complete; tile w-1 consumed
        }
        if (lane == 0) s_trades[warp] = ntr;
        __syncthreads();
    } else {
        // ---------------- the summing warp: lane j <-> individual ind0 + j ----------------
        double total = 0.0;                                                             // drl_engine.py:26
        const int j = lane < ACC_IND ? lane : 0;
        for (int64_t w = 0; w < nwin; ++w) {
            __syncthreads();
            const int n = (int)(T - w * 32 < 32 ? T - w * 32 : 32);
            const double* row = tile[w & 1][j];
            if (n == 32) {
#pragma unroll
                for (int s = 0; s < 32; ++s) total = add_rn(total, row[s]);             // drl_engine.py:54
            } else {
                for (int s = 0; s < n; ++s) total = add_rn(total, row[s]);
            }
        }
        __syncthreads();
        const int64_t ind = ind0 + lane;
        if (lane < ACC_IND && ind < count) {
            const int ntr = s_trades[lane];
            fitness[ind] = episode_fitness(total, ntr);
            trades[ind] = ntr;
        }
    }
}

}  // namespace

int launch_account(const sgmm_bundle* b, const uint64_t* codes, int64_t count, double phi, double fee, double* fitness,
                   int32_t* trades, cudaStream_t st, bool float_offsets)
{
    if (count == 0) return SGMM_OK;
    const unsigned grid = (unsigned)((count + ACC_IND - 1) / ACC_IND);
    void (*kern)(const uint64_t*, const BarPx*, int64_t, int64_t, double, double, double, double*, int32_t*) =
        fee != 0.0 ? (float_offsets ? account_kernel<true, true> : account_kernel<true, false>)
                   : (float_offsets ? account_kernel<false, true> : account_kernel<false, false>);
    kern<<<grid, ACC_THREADS, 0, st>>>(codes, b->px, b->T, count, b->tick, phi, fee, fitness, trades);
    return check_cuda(cudaGetLastError(), "account_kernel launch");
}

// The code buffer of a bundle: [count][T] 64-bit codes, grown on demand.  It is scratch of ONE rollout at a time: an eager
// rollout arriving on another stream than the last user waits for the last user's event; captured rollouts of one bundle
// must stay on one stream.  An outgrown buffer is freed, unless a capture has used the bundle's buffer (then retired).
int reserve_codes(const sgmm_bundle* cb, int64_t count, cudaStream_t st, uint64_t** out)
{
    sgmm_bundle* b = const_cast<sgmm_bundle*>(cb);
    std::lock_guard<std::mutex> lock(b->codes_mutex);
    const size_t want = (size_t)count * (size_t)b->T;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (st) cudaStreamIsCapturing(st, &cap);
    // another stream used the buffer last: order this rollout after its accounting kernel (a capture cannot wait on an
    // event recorded outside it -- captured rollouts of one bundle must stay on one stream, as the header says)
    if (b->codes_busy && b->codes_stream != st && cap == cudaStreamCaptureStatusNone && b->codes_done)
        if (int rc = check_cuda(cudaStreamWaitEvent(st, b->codes_done, 0), "cudaStreamWaitEvent(code buffer)")) return rc;
    if (cap != cudaStreamCaptureStatusNone) b->codes_captured = true;
    if (b->codes_cap < want) {
        if (cap != cudaStreamCaptureStatusNone) {
            set_error("the code buffer of the bundle holds %zu codes, this rollout needs %zu: run one rollout of this size outside "
                      "the stream capture first", b->codes_cap, want);
            return SGMM_ERR_INVALID;
        }
        // a captured CUDA graph may hold the old buffer's address: once any capture has used this bundle's code buffer the
        // outgrown buffers stay alive until the bundle is destroyed; otherwise cudaFree (which synchronises the device,
        // so every enqueued user is done) returns the memory now -- no unbounded growth when population sizes vary
        if (b->codes) { if (b->codes_captured) b->codes_retired.push_back(b->codes); else cudaFree(b->codes); }
        b->codes = nullptr; b->codes_cap = 0;
        const size_t grow = want + want / 4;
        if (int rc = check_cuda(cudaMalloc(&b->codes, grow * sizeof(uint64_t)), "cudaMalloc(code buffer)")) return rc;
        b->codes_cap = grow;
    }
    *out = b->codes;
    return SGMM_OK;
}

namespace {

// release_codes; `report` = false leaves the thread's error message alone (an error exit keeps its own message)
int release(const sgmm_bundle* cb, cudaStream_t st, bool report)
{
    sgmm_bundle* b = const_cast<sgmm_bundle*>(cb);
    std::lock_guard<std::mutex> lock(b->codes_mutex);
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (st) cudaStreamIsCapturing(st, &cap);
    if (cap != cudaStreamCaptureStatusNone) return SGMM_OK;
    auto ck = [report](cudaError_t e, const char* what) {
        return report ? check_cuda(e, what) : (e == cudaSuccess ? SGMM_OK : SGMM_ERR_CUDA);
    };
    if (!b->codes_done)
        if (int rc = ck(cudaEventCreateWithFlags(&b->codes_done, cudaEventDisableTiming), "cudaEventCreate(code buffer)")) return rc;
    if (int rc = ck(cudaEventRecord(b->codes_done, st), "cudaEventRecord(code buffer)")) return rc;
    b->codes_stream = st; b->codes_busy = true;
    return SGMM_OK;
}

}  // namespace

int release_codes(const sgmm_bundle* b, cudaStream_t st) { return release(b, st, true); }

CodesRelease::~CodesRelease()
{
    if (pending) release(b, st, false);
}

}  // namespace sgmm
