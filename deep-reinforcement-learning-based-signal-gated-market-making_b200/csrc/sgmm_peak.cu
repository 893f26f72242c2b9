// sgmm_peak.cu -- measured FP32 FMA throughput of the device: the roofline denominator of the
// H=32 rollout (SURVEY.md 8d: "the builder must measure an FFMA peak on the box").
#include "sgmm_internal.h"

namespace sgmm {

template <bool PACKED>
__global__ void __launch_bounds__(256) fma_peak_kernel(float* out, int iters, float seed)
{
    float2 acc[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) acc[i] = make_float2(seed + i, seed - i);
    const float2 m = make_float2(1.0000001f, 0.9999999f), c = make_float2(1e-7f, -1e-7f);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int i = 0; i < 12; ++i) {
                if (PACKED) acc[i] = __ffma2_rn(acc[i], m, c);
                else { acc[i].x = __fmaf_rn(acc[i].x, m.x, c.x); acc[i].y = __fmaf_rn(acc[i].y, m.y, c.y); }
            }
        }
    }
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < 12; ++i) s += acc[i].x + acc[i].y;
    if (s == 123.456f) out[0] = s;      // never true; keeps the chain alive
}

template <bool PACKED>
static int time_variant(int blocks, int iters, float* d_out, cudaStream_t st, double* tflops)
{
    cudaEvent_t e0, e1;
    if (int rc = check_cuda(cudaEventCreate(&e0), "cudaEventCreate")) return rc;
    if (int rc = check_cuda(cudaEventCreate(&e1), "cudaEventCreate")) return rc;
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0, st);
        fma_peak_kernel<PACKED><<<blocks, 256, 0, st>>>(d_out, iters, 1.0f);
        cudaEventRecord(e1, st);
        if (int rc = check_cuda(cudaEventSynchronize(e1), "fma_peak_kernel")) return rc;
        float ms = 0.f; cudaEventElapsedTime(&ms, e0, e1);
        const double flop = 2.0 * 2.0 * 12.0 * 8.0 * (double)iters * 256.0 * (double)blocks;
        const double t = flop / ((double)ms * 1e-3) / 1e12;
        if (rep > 0 && t > best) best = t;      // first repetition is warm-up
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *tflops = best;
    return SGMM_OK;
}

}  // namespace sgmm

using namespace sgmm;

extern "C" int sgmm_measure_fp32_peak(int device, double* tflops, void* stream)
{
    if (!tflops) { set_error("tflops is NULL"); return SGMM_ERR_INVALID; }
    int prev = 0; cudaGetDevice(&prev);
    if (int rc = check_cuda(cudaSetDevice(device), "cudaSetDevice")) return rc;
    const int sms = sm_count(device);
    float* d_out = nullptr;
    int rc = check_cuda(cudaMalloc(&d_out, 256), "cudaMalloc");
    double a = 0.0, b = 0.0;
    cudaStream_t st = (cudaStream_t)stream;
    if (!rc) rc = time_variant<false>(sms * 8, 4096, d_out, st, &a);
    if (!rc) rc = time_variant<true>(sms * 8, 4096, d_out, st, &b);
    cudaFree(d_out);
    cudaSetDevice(prev);
    *tflops = a > b ? a : b;
    return rc;
}
