// Chip-wide issue-rate probes for the roofline denominators MEASURED_PEAKS.json lacks
// (SURVEY.md section 8d): MUFU.EX2 results/s and FFMA/s.  Eight independent dependent-chains
// per thread keep each pipe saturated; 8 CTAs of 256 threads per SM fill every scheduler.
#include "tc_common.cuh"
#include "../../include/dgvcc_b200.h"

namespace dgvcc {

constexpr int PROBE_THREADS = 256;
constexpr int PROBE_CHAINS = 8;

__global__ void __launch_bounds__(PROBE_THREADS) probe_ex2_kernel(float* sink, int iters) {
    float v[PROBE_CHAINS];
#pragma unroll
    for (int c = 0; c < PROBE_CHAINS; ++c) v[c] = -1e-3f * (float)(threadIdx.x + c);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int c = 0; c < PROBE_CHAINS; ++c) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(v[c]));
    }
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < PROBE_CHAINS; ++c) s += v[c];
    if (s == 123.456f) sink[0] = s;  // keeps the chains alive, never true in practice
}

__global__ void __launch_bounds__(PROBE_THREADS) probe_ffma_kernel(float* sink, int iters) {
    float v[PROBE_CHAINS];
    const float a = 0.999f, b = 1e-3f;
#pragma unroll
    for (int c = 0; c < PROBE_CHAINS; ++c) v[c] = (float)(threadIdx.x + c);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int c = 0; c < PROBE_CHAINS; ++c) asm volatile("fma.rn.f32 %0, %0, %1, %2;" : "+f"(v[c]) : "f"(a), "f"(b));
    }
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < PROBE_CHAINS; ++c) s += v[c];
    if (s == 123.456f) sink[0] = s;
}

// Tensor-pipe probe: every SM issues back-to-back tcgen05.mma.kind::tf32 (M = 128, N = 256, K = 8; A and B K-major
// 128B-swizzled tiles in shared memory, fp32 accumulators in 256 TMEM columns) from one thread, the way the ISW
// Gram kernel does.  N = 256 keeps the operand traffic (12 KB per MMA) under the SM's shared-memory bandwidth, so
// the measured rate is the tensor pipe's own: the denominator of the Gram's roofline (MEASURED_PEAKS.json has bf16 only).
constexpr int TF32_PROBE_SMEM = 16384 + 32768 + 1024 + 64;

__global__ void __launch_bounds__(128, 1) probe_tf32_kernel(float* sink, int iters) {
    using namespace dgvcc::tc;
    extern __shared__ uint8_t probe_smem[];
    const uint32_t base = (smem_u32(probe_smem) + 1023u) & ~1023u;
    uint8_t* base_ptr = probe_smem + (base - smem_u32(probe_smem));
    const uint32_t bar = base + 16384 + 32768;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(base_ptr + 16384 + 32768 + 16);
    float* tiles = reinterpret_cast<float*>(base_ptr);
    for (int i = threadIdx.x; i < (16384 + 32768) / 4; i += blockDim.x)
        tiles[i] = 1.0f + 1e-3f * (float)((i * 2654435761u) >> 22);  // finite, non-trivial operand bits
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(256) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;
    if (threadIdx.x == 0) {
        constexpr uint32_t idesc = umma_idesc_tf32(128, 256, false);
        const uint64_t a = umma_desc_sw128(base, 16, 1024), b = umma_desc_sw128(base + 16384, 16, 1024);
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) umma_tf32(tmem_d, a + 2 * ks, b + 2 * ks, idesc, (it | ks) != 0);
        }
        umma_commit(bar);
        mbar_wait(bar, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t r[32];
        tmem_ld32(tmem_d, r);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (__uint_as_float(r[0]) == 123.456f) sink[0] = 1.f;  // keeps the accumulator observable
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(256) : "memory");
    }
}

// ex2.approx.ftz.f32 and ex2_fma of every t[i]; ex2_fma takes the values two at a time, like the sweeps' row pairs.
__global__ void __launch_bounds__(256) probe_ex2_fma_kernel(const float* __restrict__ t, int n, float* __restrict__ mufu,
                                                            float* __restrict__ fma) {
    const int64_t i = 2 * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
    if (i >= n) return;
    const bool pair = i + 1 < n;
    const float t0 = t[i], t1 = pair ? t[i + 1] : t0;
    float e0, e1;
    unpack2(ex2_fma(pack2(t0, t1)), e0, e1);
    mufu[i] = ex2_ftz(t0);
    fma[i] = e0;
    if (pair) {
        mufu[i + 1] = ex2_ftz(t1);
        fma[i + 1] = e1;
    }
}

static int probe_grid() {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms * 8;
}

}  // namespace dgvcc

extern "C" int dgvcc_probe_ex2(float* sink, int iters, int64_t* ops_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!sink || iters <= 0) return DGVCC_ERR_ARG;
    const int grid = dgvcc::probe_grid();
    dgvcc::probe_ex2_kernel<<<grid, dgvcc::PROBE_THREADS, 0, (cudaStream_t)stream>>>(sink, iters);
    if (ops_out) *ops_out = (int64_t)grid * dgvcc::PROBE_THREADS * dgvcc::PROBE_CHAINS * iters;
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_probe_ffma(float* sink, int iters, int64_t* ops_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!sink || iters <= 0) return DGVCC_ERR_ARG;
    const int grid = dgvcc::probe_grid();
    dgvcc::probe_ffma_kernel<<<grid, dgvcc::PROBE_THREADS, 0, (cudaStream_t)stream>>>(sink, iters);
    if (ops_out) *ops_out = (int64_t)grid * dgvcc::PROBE_THREADS * dgvcc::PROBE_CHAINS * iters;
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_probe_ex2_fma(const float* t, int n, float* mufu_out, float* fma_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!t || !mufu_out || !fma_out || n <= 0) return DGVCC_ERR_ARG;
    const int grid = (int)(((int64_t)n + 511) / 512);
    dgvcc::probe_ex2_fma_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(t, n, mufu_out, fma_out);
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_probe_tf32(float* sink, int iters, int64_t* flops_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!sink || iters <= 0) return DGVCC_ERR_ARG;
    static dgvcc::PerDeviceOnce once;
    if (once.first())
        DGVCC_RETURN_IF_CUDA(cudaFuncSetAttribute(dgvcc::probe_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                  dgvcc::TF32_PROBE_SMEM));
    const int grid = dgvcc::probe_grid() / 8;  // one CTA per SM
    dgvcc::probe_tf32_kernel<<<grid, 128, dgvcc::TF32_PROBE_SMEM, (cudaStream_t)stream>>>(sink, iters);
    if (flops_out) *flops_out = (int64_t)grid * iters * 4 * (2LL * 128 * 256 * 8);
    return (int)cudaGetLastError();
}
