// Shared device helpers for the dgvcc_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define DGVCC_OK 0
#define DGVCC_ERR_ARG (-1)        // bad argument (null pointer, non-positive size ...)
#define DGVCC_ERR_WORKSPACE (-2)  // caller-owned workspace too small
#define DGVCC_ERR_UNSUPPORTED (-3)

#define DGVCC_RETURN_IF_CUDA(expr)            \
    do {                                      \
        cudaError_t _e = (expr);              \
        if (_e != cudaSuccess) return (int)_e; \
    } while (0)

// Checked build (`DGVCC_BOUNDS_CHECK=1 python -m dgvcc_b200.build`, nvcc -DDGVCC_BOUNDS_CHECK; loaded instead of the
// product library when the same variable is set at import): every index that comes out of a host-built table or a
// data-dependent computation is tested where it is used; a violation is a device-side assert (site, block, thread
// and condition are reported, the launch fails with cudaErrorAssert) instead of silent memory corruption.
// compute-sanitizer is closed on the GPU pool this was built on -- this is its substitute.  The product build
// compiles every check away (the condition is not evaluated; `cuobjdump -sass` of the objects is identical with and
// without the DGVCC_DEV_CHECK lines).
#ifdef DGVCC_BOUNDS_CHECK
#undef NDEBUG
#include <assert.h>
// device-side assert: the runtime reports file, line, block, thread and the condition when the context is torn down
#define DGVCC_DEV_CHECK(cond) assert(cond)
#define DGVCC_BOUNDS_CHECKED 1
#else
#define DGVCC_DEV_CHECK(cond) ((void)0)
#define DGVCC_BOUNDS_CHECKED 0
#endif

namespace dgvcc {

// Every launcher runs on the device that owns the caller's stream, whatever the calling thread's current
// device is (the reference's configs pass device='cuda:1' etc. without ever calling set_device); the
// previous current device is restored on return.
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(void* stream) {
        int cur = 0, want = 0;
        // A stream that is being captured into a CUDA graph belongs to the current device (the capture was begun on it),
        // and cudaStreamGetDevice is one of the calls a global-mode capture forbids: asking would invalidate the graph.
        cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing((cudaStream_t)stream, &capturing) != cudaSuccess) { (void)cudaGetLastError(); return; }
        if (capturing != cudaStreamCaptureStatusNone) return;
        if (cudaGetDevice(&cur) != cudaSuccess) return;
        if (cudaStreamGetDevice((cudaStream_t)stream, &want) != cudaSuccess) { (void)cudaGetLastError(); return; }
        if (want != cur && cudaSetDevice(want) == cudaSuccess) prev = cur;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define DGVCC_DEVICE_GUARD(stream) ::dgvcc::DeviceGuard dgvcc_device_guard_(stream)

// Function attributes (opt-in dynamic shared memory) are per device: `static PerDeviceOnce once;`
// `if (once.first()) cudaFuncSetAttribute(...)` configures a kernel the first time each device launches it.
struct PerDeviceOnce {
    bool done[64] = {};
    bool first() {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return true;
        if (done[d]) return false;
        done[d] = true;  // a race only repeats the same idempotent call
        return true;
    }
};

constexpr unsigned FULL_MASK = 0xffffffffu;
constexpr float LOG2E = 1.4426950408889634f;

// One MUFU.EX2; results below 2^-126 flush to zero (posteriors < 1.2e-38, far under the 1e-30 atol).
__device__ __forceinline__ float ex2_ftz(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Two fp32 values in one 64-bit register: Blackwell's packed add/mul/fma.f32x2 (SASS FADD2 / FMUL2 / FFMA2)
// do the work of two scalar instructions in one issue slot; each lane is an ordinary IEEE round-to-nearest op.
typedef unsigned long long f2;
__device__ __forceinline__ f2 pack2(float lo, float hi) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(f2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { f2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { f2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

// t clamped to [-127, 128]; NaN stays NaN (max.NaN / min.NaN, where fmaxf / fminf would return the bound).
__device__ __forceinline__ float ex2_fma_clamp(float t) {
    float r;
    asm("max.NaN.f32 %0, %1, 0fC2FE0000;\n\tmin.NaN.f32 %0, %0, 0f43000000;" : "=f"(r) : "f"(t));
    return r;
}

// 2^t for both lanes on the FMA and ALU pipes only, a stand-in for ex2_ftz wherever MUFU is the bottleneck.
// t = n + f with n = RN(t) (the 1.5 * 2^23 trick: no F2I, which would share MUFU's pipe) and f in [-0.5, 0.5];
// 2^f is a degree-6 polynomial with p(0) = 1 (relative minimax, error 3.9e-9, fp32 coefficients), evaluated by Horner
// in FFMA2; 2^n is built in the exponent field and applied by one flush-to-zero multiply.  Like ex2.approx.ftz.f32:
//   * the result is +0 exactly for t < -126: n = -127 gives the factor +0, and n = -126 with f < 0 gives a subnormal
//     that the multiply flushes -- the zero set ExpCull relies on;
//   * NaN gives NaN, -inf gives +0, +inf gives +inf, 2^n is exact for integer t;
//   * max relative error over every fp32 t in [-126, 0] is 7.8e-8 (MUFU.EX2: 1.4e-7), see profiles/r3_bl_fma_exp.md.
// For t > 127.5 it returns +inf where MUFU still returns a finite value; exponents of the loss are <= 2^-8.
__device__ __forceinline__ f2 ex2_fma(f2 t) {
    float t0, t1;
    unpack2(t, t0, t1);
    const f2 tc = pack2(ex2_fma_clamp(t0), ex2_fma_clamp(t1));
    const f2 fi = add2(tc, pack2(12582912.f, 12582912.f));   // n in the low mantissa bits
    const f2 n = add2(fi, pack2(-12582912.f, -12582912.f));  // exact
    const f2 f = fma2(n, pack2(-1.f, -1.f), tc);              // exact
    f2 p = pack2(1.54697322e-4f, 1.54697322e-4f);
    p = fma2(p, f, pack2(1.34100008e-3f, 1.34100008e-3f));
    p = fma2(p, f, pack2(9.61803086e-3f, 9.61803086e-3f));
    p = fma2(p, f, pack2(5.55029735e-2f, 5.55029735e-2f));
    p = fma2(p, f, pack2(2.40226507e-1f, 2.40226507e-1f));
    p = fma2(p, f, pack2(6.93147242e-1f, 6.93147242e-1f));
    p = fma2(p, f, pack2(1.f, 1.f));
    float fi0, fi1;
    unpack2(fi, fi0, fi1);
    // (n + 127) << 23: the low bits of fi hold n in two's complement; n = 128 gives +inf, n = -127 gives +0
    const f2 s = pack2(__int_as_float((__float_as_int(fi0) << 23) + 0x3f800000),
                       __int_as_float((__float_as_int(fi1) << 23) + 0x3f800000));
    f2 r;
    asm("mul.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(p), "l"(s));
    return r;
}

// ex2_fma on one lane with the same operations (fma.rn / add.rn / mul.rn.ftz are IEEE per lane)
__device__ __forceinline__ float ex2_fma1(float t) {
    const float tc = ex2_fma_clamp(t);
    const float fi = __fadd_rn(tc, 12582912.f);
    const float n = __fadd_rn(fi, -12582912.f);
    const float f = __fmaf_rn(n, -1.f, tc);
    float p = 1.54697322e-4f;
    p = __fmaf_rn(p, f, 1.34100008e-3f);
    p = __fmaf_rn(p, f, 9.61803086e-3f);
    p = __fmaf_rn(p, f, 5.55029735e-2f);
    p = __fmaf_rn(p, f, 2.40226507e-1f);
    p = __fmaf_rn(p, f, 6.93147242e-1f);
    p = __fmaf_rn(p, f, 1.f);
    const float s = __int_as_float((__float_as_int(fi) << 23) + 0x3f800000);
    float r;
    asm("mul.rn.ftz.f32 %0, %1, %2;" : "=f"(r) : "f"(p), "f"(s));
    return r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
    return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
    return v;
}

__host__ __device__ __forceinline__ int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ __forceinline__ size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace dgvcc
