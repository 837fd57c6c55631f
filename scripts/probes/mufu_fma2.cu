// Microbenchmark 4: the 8x2 inner loop of bl_z_kernel (staged xs / yd loads from shared memory, FADD2 + FFMA2
// argument, FADD2 accumulation, 4 CTAs of 128 threads per SM) with a share of its exponentials moved from MUFU.EX2 to
// ex2_fma, a packed FMA-pipe exponential with MUFU's zero set and better accuracy (below):
//   share 0   : every exponential on MUFU
//   share 1/8 : the row-7 lane of the last row pair on a scalar copy of ex2_fma's arithmetic
//   share 1/4 : the whole last row pair (rows 6, 7) on the packed ex2_fma
// Then the accuracy table of ex2_fma against ex2.approx.ftz.f32, both measured against fp64 exp2 over every fp32 t in
// [-130, 2^-8], and the special values.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o mufu_fma2 scripts/probes/mufu_fma2.cu
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cuda_runtime.h>

__device__ __forceinline__ float ex2_ftz(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// Two fp32 values in one 64-bit register: Blackwell's packed add/mul/fma.f32x2 (SASS FADD2 / FMUL2 / FFMA2)
// do the work of two scalar instructions in one issue slot; each lane is an ordinary IEEE round-to-nearest op.
typedef unsigned long long f2;
__device__ __forceinline__ f2 pack2(float lo, float hi) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(f2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
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

constexpr int R = 8, C = 2, TILE = 128;

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

template <int SHARE>  // 0, 1 (= 1/8), 2 (= 1/4)
__device__ __forceinline__ f2 exp_pair(f2 t, int q) {
    if (SHARE == 2 && q == R / 2 - 1) return ex2_fma(t);
    float t0, t1;
    unpack2(t, t0, t1);
    if (SHARE == 1 && q == R / 2 - 1) return pack2(ex2_ftz(t0), ex2_fma1(t1));
    return pack2(ex2_ftz(t0), ex2_ftz(t1));
}

struct __align__(16) Tile {
    float2 xs[TILE];
    float yd[TILE][R];
};

template <int SHARE>
__global__ void __launch_bounds__(128, 4) sweep(float* out, int reps, float k1) {
    __shared__ Tile tiles[4];
    Tile& tile = tiles[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    // points scattered over a 1024 x 768 image, pixel tile near its middle: a spread of exponents down to below -126
    for (int i = lane; i < TILE; i += 32) {
        const float x = (float)((i * 37 + blockIdx.x * 13) % 1024), y = (float)((i * 53 + blockIdx.x * 7) % 768);
        tile.xs[i] = make_float2(x, x * x);
        for (int r = 0; r < R; ++r) {
            const float cy = 380.f + 8.f * r;
            tile.yd[i][r] = (y - cy) * (y - cy);
        }
    }
    __syncwarp();
    const float cx0 = 8.f * (lane + 32 * (blockIdx.x & 3)) + 4.f;
    float cxm2[C], cxx[C];
    for (int c = 0; c < C; ++c) { const float cx = cx0 + 256.f * c; cxm2[c] = -2.f * cx; cxx[c] = cx * cx; }
    f2 zp[R / 2][C], k2p[R / 2][C];
    const f2 k1p = pack2(k1, k1);
#pragma unroll
    for (int q = 0; q < R / 2; ++q)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            zp[q][c] = pack2(0.f, 0.f);
            k2p[q][c] = pack2(1e-3f * q, 2e-3f * c);
        }
    for (int rep = 0; rep < reps; ++rep) {
#pragma unroll 2
        for (int i = 0; i < TILE; ++i) {
            const float2 xs = tile.xs[i];
            f2 yd[R / 2];
#pragma unroll
            for (int q = 0; q < R / 4; ++q) {
                const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&tile.yd[i][4 * q]);
                yd[2 * q] = v.x; yd[2 * q + 1] = v.y;
            }
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float xd = __fadd_rn(__fadd_rn(__fmul_rn(xs.x, cxm2[c]), xs.y), cxx[c]);
                const f2 xd2 = pack2(xd, xd);
#pragma unroll
                for (int q = 0; q < R / 2; ++q)
                    zp[q][c] = add2(zp[q][c], exp_pair<SHARE>(fma2(add2(yd[q], xd2), k1p, k2p[q][c]), q));
            }
        }
    }
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < R / 2; ++q)
#pragma unroll
        for (int c = 0; c < C; ++c) { float a, b; unpack2(zp[q][c], a, b); s += a + b; }
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <int SHARE>
float time_sweep(float* out, int grid, int reps, float k1) {
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    sweep<SHARE><<<grid, 128>>>(out, reps, k1);
    cudaEventRecord(a);
    for (int i = 0; i < 5; ++i) sweep<SHARE><<<grid, 128>>>(out, reps, k1);
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a); cudaEventDestroy(b);
    return ms / 5;
}

// Accuracy over every fp32 t in [-130, 2^-8] (two bit-pattern ranges: -0 .. -130 and +0 .. 2^-8).
struct Stats {
    unsigned int mufu_err, fma_err;        // max relative error (float bits) with 2^t >= 2^-126, t <= 0
    unsigned int mufu_err_all, fma_err_all;  // same over the whole range up to 2^-8
    unsigned long long zero_mismatch, fma_nonpos_zero, lane_mismatch, mufu_below_zero, n;
    unsigned int worst_fma_t, worst_mufu_t;
};

__device__ void err_one(float t, float m, float e, Stats* st, float& wm, float& we, float& wma, float& wea, float& tm,
                        float& te, unsigned long long& zm, unsigned long long& bad0) {
    const double ref = exp2((double)t);
    if ((m == 0.f) != (e == 0.f) || __float_as_uint(e) == 0x80000000u) ++zm;
    if (t < -126.f && __float_as_uint(e) != 0u) ++bad0;
    if (t >= -126.f) {
        const float rm = (float)fabs(((double)m - ref) / ref), re = (float)fabs(((double)e - ref) / ref);
        wma = fmaxf(wma, rm);
        wea = fmaxf(wea, re);
        if (t <= 0.f) {
            if (rm > wm) { wm = rm; tm = t; }
            if (re > we) { we = re; te = t; }
        }
    }
}

__global__ void err_kernel(Stats* st, unsigned int lo, unsigned int hi) {
    float wm = 0.f, we = 0.f, wma = 0.f, wea = 0.f, tm = 0.f, te = 0.f;
    unsigned long long zm = 0, bad0 = 0, lanes = 0, mz = 0, cnt = 0;
    const unsigned int stride = gridDim.x * blockDim.x * 2;
    for (unsigned long long u = lo + 2ull * (blockIdx.x * blockDim.x + threadIdx.x); u <= hi; u += stride) {
        const float t0 = __uint_as_float((unsigned int)u);
        const float t1 = u + 1 <= hi ? __uint_as_float((unsigned int)u + 1) : t0;
        float e0, e1;
        unpack2(ex2_fma(pack2(t0, t1)), e0, e1);
        if (__float_as_uint(e0) != __float_as_uint(ex2_fma1(t0)) || __float_as_uint(e1) != __float_as_uint(ex2_fma1(t1)))
            ++lanes;
        const float m0 = ex2_ftz(t0), m1 = ex2_ftz(t1);
        if (t0 >= -126.f && m0 == 0.f) ++mz;
        err_one(t0, m0, e0, st, wm, we, wma, wea, tm, te, zm, bad0);
        ++cnt;
        if (u + 1 <= hi) { err_one(t1, m1, e1, st, wm, we, wma, wea, tm, te, zm, bad0); ++cnt; }
    }
    if (wm > __uint_as_float(atomicMax(&st->mufu_err, __float_as_uint(wm)))) st->worst_mufu_t = __float_as_uint(tm);
    if (we > __uint_as_float(atomicMax(&st->fma_err, __float_as_uint(we)))) st->worst_fma_t = __float_as_uint(te);
    atomicMax(&st->mufu_err_all, __float_as_uint(wma));
    atomicMax(&st->fma_err_all, __float_as_uint(wea));
    atomicAdd(&st->zero_mismatch, zm);
    atomicAdd(&st->fma_nonpos_zero, bad0);
    atomicAdd(&st->lane_mismatch, lanes);
    atomicAdd(&st->mufu_below_zero, mz);
    atomicAdd(&st->n, cnt);
}

__global__ void special_kernel(const float* t, float* m, float* e, int n) {
    const int i = threadIdx.x;
    if (i < n) {
        m[i] = ex2_ftz(t[i]);
        float lo, hi;
        unpack2(ex2_fma(pack2(t[i], 0.f)), lo, hi);
        e[i] = lo;
    }
}

static unsigned int bits(float f) { unsigned int u; memcpy(&u, &f, 4); return u; }
static float flt(unsigned int u) { float f; memcpy(&f, &u, 4); return f; }

int main() {
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, 0);
    printf("device %s, %d SMs\n", prop.name, prop.multiProcessorCount);

    // ---- accuracy table
    Stats* st;
    cudaMallocManaged(&st, sizeof(Stats));
    memset(st, 0, sizeof(Stats));
    err_kernel<<<prop.multiProcessorCount * 8, 256>>>(st, 0x80000000u, bits(-130.f));  // -0 .. -130
    err_kernel<<<prop.multiProcessorCount * 8, 256>>>(st, 0x00000000u, bits(0.00390625f));  // +0 .. 2^-8
    cudaDeviceSynchronize();
    printf("accuracy over every fp32 t in [-130, 2^-8] (%llu values), relative error against fp64 exp2:\n", st->n);
    printf("  t in [-126, 0]      : MUFU.EX2 max %.3e (at t = %.9g)   ex2_fma max %.3e (at t = %.9g)\n",
           flt(st->mufu_err), flt(st->worst_mufu_t), flt(st->fma_err), flt(st->worst_fma_t));
    printf("  t in [-126, 2^-8]   : MUFU.EX2 max %.3e                   ex2_fma max %.3e\n", flt(st->mufu_err_all),
           flt(st->fma_err_all));
    printf("  zero sets differ at %llu values; ex2_fma != +0 below -126 at %llu; MUFU zero at t >= -126: %llu\n",
           st->zero_mismatch, st->fma_nonpos_zero, st->mufu_below_zero);
    printf("  packed lanes != scalar copy at %llu values\n", st->lane_mismatch);

    const float sp[] = {NAN, -NAN, INFINITY, -INFINITY, -0.f, 0.f, -126.f, -126.00001f, -126.5f, -127.f, -128.f,
                        -1e30f, 1.f, 0.00390625f, -1.f, -0.5f, 127.f};
    const int ns = sizeof(sp) / sizeof(sp[0]);
    float *dt, *dm, *de;
    cudaMallocManaged(&dt, sizeof(sp)); cudaMallocManaged(&dm, sizeof(sp)); cudaMallocManaged(&de, sizeof(sp));
    memcpy(dt, sp, sizeof(sp));
    special_kernel<<<1, 32>>>(dt, dm, de, ns);
    cudaDeviceSynchronize();
    printf("special values (t: MUFU.EX2 / ex2_fma, bits):\n");
    for (int i = 0; i < ns; ++i)
        printf("  %-12g: %-12g %08x / %-12g %08x %s\n", sp[i], dm[i], bits(dm[i]), de[i], bits(de[i]),
               bits(dm[i]) == bits(de[i]) || (std::isnan(dm[i]) && std::isnan(de[i])) ? "" : "(differs)");

    // ---- throughput of the 8x2 loop
    const int grid = prop.multiProcessorCount * 4 * 8, reps = 64;
    float* out;
    cudaMalloc(&out, (size_t)grid * 128 * sizeof(float));
    const double exps = (double)grid * 128 * reps * TILE * R * C;
    const float k1 = -1.4426950408889634f / 128.f;  // sigma = 8: 2 sigma^2 = 128
    for (int round = 0; round < 3; ++round) {
        const float t0 = time_sweep<0>(out, grid, reps, k1);
        const float t1 = time_sweep<1>(out, grid, reps, k1);
        const float t2 = time_sweep<2>(out, grid, reps, k1);
        printf("round %d: share 0: %.3f ms (%.2f Texp/s)  share 1/8: %.3f ms (x%.3f)  share 1/4: %.3f ms (x%.3f)  %s\n",
               round, t0, exps / t0 / 1e9, t1, t0 / t1, t2, t0 / t2, cudaGetErrorString(cudaGetLastError()));
    }
    return 0;
}
