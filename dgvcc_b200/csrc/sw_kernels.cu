// Switchable whitening for sm_100a (SURVEY.md section 8f, rank 4).
//
// Replaces SwitchWhiten2d.forward (models/ISW/switchwhiten.py:84-183) and SyncMeanCov / SyncSwitchWhiten2d.forward
// (models/ISW/sync_switchwhiten.py:9-56,135-223).  The evaluation order is the one oracle/switchwhiten_oracle.py:
// ``decomposed`` spells out:
//
//   forward   moments pass     one read of x: sums and upper-triangular products per (sample, group), shifted by a
//                              sample mean of the plane
//             instance stats   mean_in, cov_in (fp64)
//             batch mean/cov   from the per-sample statistics (the caller exchanges them between ranks)
//             whiten matrices  softmax mix, T Newton iterations on cp x cp matrices in fp64, A = diag(weight) wm
//             affine pass      y = A x + cst, one read of x, one write of y
//   backward  moments pass     one read of x and grad_y: K = sum_p gy (x - mean_in)^T, s = sum_p gy
//             matrices         closed-form adjoint of the Newton iteration -> d loss / d cov, d loss / d mean
//             reductions       over samples (batch statistics, weights) and over groups (layer statistics)
//             coefficients     M1 = A^T, M2 = S_in + S_bn, cst
//             affine pass      grad_x = M1 grad_y + M2 x + cst, one read of x and grad_y, one write
//
// The two affine passes and the two moments passes are HBM-bound (8 / 12 bytes per element against 16 / 32 FMAs for
// cp = 16); the matrix kernels touch a few KB per (sample, group) and run in fp64 so that the fp32 rounding of the
// reference's own Newton iteration is the only difference that parity has to absorb.
#include "common.cuh"
#include "../../include/dgvcc_b200.h"

namespace dgvcc {
namespace sw {

constexpr int MOM_THREADS = 128;
constexpr int NUM_SMS = 148;         // B200
constexpr int MAX_DEVICES = 64;
constexpr int MOM_CTAS_PER_SM = 2;   // ~210 registers x 128 threads
constexpr int MAT_THREADS = 256;     // one thread per entry of a 16 x 16 matrix
constexpr int AFF_THREADS = 128;
constexpr int MAX_T = DGVCC_SW_MAX_T;
constexpr int BWD_ROWS = 8;          // rows of K per backward-moments CTA (register budget)

enum Dot { D_COV_BN = 0, D_COV_IN, D_DIAG_BN, D_DIAG_IN, D_TR, D_TR_VARLN, D_MEAN_BN, D_MEAN_IN, D_SUM_GMEAN,
           D_GMEAN_MEANLN, N_DOTS };
enum Ln { L_MEAN = 0, L_VAR, L_G_VAR, L_G_MEAN, N_LN };

struct Mix {
    double a_bn, a_in, a_ln;   // mean coefficients
    double b_bn, b_in, b_ln;   // covariance coefficients
    double d_bn, d_in;         // diagonal-only covariance coefficients (sw_type 5)
    double mw[5], vw[5];
};

__device__ __forceinline__ void softmax_small(const float* logits, int k, double* out) {
    double m = -1e300, s = 0.0;
    for (int i = 0; i < k; ++i) m = fmax(m, (double)logits[i]);
    for (int i = 0; i < k; ++i) { out[i] = exp((double)logits[i] - m); s += out[i]; }
    for (int i = 0; i < k; ++i) out[i] /= s;
}

// switchwhiten.py:137-164
__device__ __forceinline__ Mix mix_coeffs(int sw_type, const float* mean_logits, const float* var_logits) {
    Mix m;
    for (int i = 0; i < 5; ++i) m.mw[i] = m.vw[i] = 0.0;
    softmax_small(mean_logits, sw_type, m.mw);
    if (var_logits) softmax_small(var_logits, sw_type, m.vw);
    else for (int i = 0; i < sw_type; ++i) m.vw[i] = m.mw[i];
    if (sw_type == 2) {
        m.a_bn = m.mw[0]; m.a_in = m.mw[1]; m.a_ln = 0.0;
        m.b_bn = m.vw[0]; m.b_in = m.vw[1]; m.b_ln = 0.0; m.d_bn = m.d_in = 0.0;
    } else if (sw_type == 3) {
        m.a_bn = m.mw[0]; m.a_in = m.mw[1]; m.a_ln = m.mw[2];
        m.b_bn = m.vw[0]; m.b_in = m.vw[1]; m.b_ln = m.vw[2]; m.d_bn = m.d_in = 0.0;
    } else {
        m.a_bn = m.mw[0] + m.mw[2]; m.a_in = m.mw[1] + m.mw[3]; m.a_ln = m.mw[4];
        m.b_bn = m.vw[0]; m.b_in = m.vw[1]; m.b_ln = m.vw[4]; m.d_bn = m.vw[0]; m.d_in = m.vw[1];
    }
    return m;
}

// Sum over the 256 threads of a matrix CTA, returned to every thread.  ``red`` holds 8 doubles.
__device__ __forceinline__ double block_sum(double v, double* red) {
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < MAT_THREADS / 32; ++w) s += red[w];
    __syncthreads();
    return s;
}

__host__ __device__ __forceinline__ int tri_index(int cp, int i, int j) {  // i <= j, row-major upper triangle
    return i * cp - i * (i - 1) / 2 + (j - i);
}

// ------------------------------------------------------------------------------------------------ moments (fwd)

// The two moments passes keep ~150 accumulators per thread, so only 8 warps fit on an SM: register-staged loads
// cannot cover the HBM latency.  Each thread instead streams ITS OWN pixels through a private ring of shared-memory
// slots with 4-byte cp.async (any alignment, no barrier needed: a thread only ever reads what it copied itself).
__device__ __forceinline__ void cp_async_f32(float* smem_dst, const float* gsrc) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int FWD_STAGES = 8, BWD_STAGES = 6;   // 64 / 72 KB of dynamic shared memory per CTA for cp = 16

// Sums NV per-thread values over the lanes of a warp with a halving butterfly: 31 shuffles per 32 values instead of
// 5 per value.  Afterwards lane l holds the warp totals of values l, 32 + l, ... in out[0], out[1], ...
template <int NV>
__device__ __forceinline__ void warp_transpose_sum(const float (&acc)[NV], float (&out)[(NV + 31) / 32]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int g = 0; g < (NV + 31) / 32; ++g) {
        float v[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] = g * 32 + k < NV ? acc[g * 32 + k] : 0.f;
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            const bool up = (lane & off) != 0;
#pragma unroll
            for (int k = 0; k < off; ++k) {
                const float keep = up ? v[k + off] : v[k];
                const float send = up ? v[k] : v[k + off];
                v[k] = keep + __shfl_xor_sync(FULL_MASK, send, off);
            }
        }
        out[g] = v[0];
    }
}

// Floats per (sample, group, split) in the forward partials: the shifted sums, the upper triangle of the shifted
// products, then the shift itself.
template <int CP>
__host__ __device__ constexpr int fwd_part_floats() { return CP + CP * (CP + 1) / 2 + CP; }

// The shift the forward moments are centred on: the mean of up to 128 pixels of the plane, summed in a fixed order so
// that every CTA of a plane computes the same bits.  Centring on a sample mean rather than on one pixel keeps the
// shifted sums small when some pixels sit far from the plane mean (zero-padded corners of conv features):
// S2 / hw - delta delta^T then cancels no digits.  The sample is 16 runs of 8 consecutive pixels starting at
// (c hw) / 16, c = 0 .. 15 (every pixel when hw <= 128): a warp's load touches 4 to 8 sectors where 32 scattered
// pixels touched 32, which measured 15 % of the moments kernel's time at the benchmark shapes.
template <int CP>
__device__ __forceinline__ void sample_shift(const float* base, int hw, float (&shift)[CP], float (*sred)[CP]) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int p = hw > MOM_THREADS ? (int)(((long long)(tid >> 3) * hw) / 16) + (tid & 7) : tid;
    float v[CP], tot[1];
#pragma unroll
    for (int j = 0; j < CP; ++j) v[j] = p < hw ? __ldg(base + (size_t)j * hw + p) : 0.f;
    warp_transpose_sum<CP>(v, tot);
    if (lane < CP) sred[warp][lane] = tot[0];
    __syncthreads();
    const float inv = 1.f / (float)(hw < MOM_THREADS ? hw : MOM_THREADS);   // 2^-7 but on planes under 128 pixels
#pragma unroll
    for (int j = 0; j < CP; ++j) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < MOM_THREADS / 32; ++w) s += sred[w][j];
        shift[j] = s * inv;
    }
}

// grid (splits, n * groups).  part[(ng * splits + split) * fwd_part_floats<CP>() + k]: k < CP the shifted sums, then
// the upper triangle, then the CP shifts (the same in every split of a plane).
template <int CP>
__global__ void __launch_bounds__(MOM_THREADS, 2)
sw_moments_kernel(const float* __restrict__ x, int hw, int chunk, float* __restrict__ part) {
    constexpr int NV = CP + CP * (CP + 1) / 2;
    extern __shared__ float ring_raw[];
    float (*ring)[CP][MOM_THREADS] = reinterpret_cast<float (*)[CP][MOM_THREADS]>(ring_raw);
    __shared__ float red[MOM_THREADS / 32][NV];
    __shared__ float sred[MOM_THREADS / 32][CP];
    const float* base = x + (size_t)blockIdx.y * CP * hw;
    const int tid = threadIdx.x;
    float shift[CP], acc[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) acc[k] = 0.f;
    const int p0 = blockIdx.x * chunk, p1 = min(hw, p0 + chunk);
    const int iters = ceil_div(p1 - p0, MOM_THREADS);
    auto issue = [&](int it) {
        const int p = p0 + it * MOM_THREADS + tid;
        if (it < iters && p < p1) {
#pragma unroll
            for (int j = 0; j < CP; ++j) cp_async_f32(&ring[it % FWD_STAGES][j][tid], base + (size_t)j * hw + p);
        }
        cp_async_commit();
    };
    for (int it = 0; it < FWD_STAGES - 1; ++it) issue(it);
    sample_shift<CP>(base, hw, shift, sred);   // after the ring's first copies: their latencies overlap
    for (int it = 0; it < iters; ++it) {
        issue(it + FWD_STAGES - 1);       // its slot was read (into registers) one iteration ago
        cp_async_wait<FWD_STAGES - 1>();
        const bool valid = p0 + it * MOM_THREADS + tid < p1;
        float u[CP];
#pragma unroll
        for (int j = 0; j < CP; ++j) u[j] = valid ? ring[it % FWD_STAGES][j][tid] - shift[j] : 0.f;
        int k = CP;
#pragma unroll
        for (int i = 0; i < CP; ++i) {
            acc[i] += u[i];
#pragma unroll
            for (int j = i; j < CP; ++j, ++k) acc[k] = fmaf(u[i], u[j], acc[k]);
        }
    }
    const int warp = tid >> 5, lane = tid & 31;
    float tot[(NV + 31) / 32];
    warp_transpose_sum<NV>(acc, tot);
#pragma unroll
    for (int g = 0; g < (NV + 31) / 32; ++g)
        if (g * 32 + lane < NV) red[warp][g * 32 + lane] = tot[g];
    __syncthreads();
    float* out = part + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * fwd_part_floats<CP>();
    for (int k = tid; k < NV; k += MOM_THREADS) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < MOM_THREADS / 32; ++w) s += red[w][k];
        out[k] = s;
    }
    if (tid < CP) {
#pragma unroll
        for (int j = 0; j < CP; ++j)
            if (j == tid) out[NV + j] = shift[j];   // static register index: no local-memory copy of shift
    }
}

// grid n * groups, 256 threads.
template <int CP>
__global__ void __launch_bounds__(MAT_THREADS)
sw_instance_stats_kernel(const float* __restrict__ part, int splits, int hw, double* __restrict__ mean_in,
                         double* __restrict__ cov_in) {
    constexpr int NV = CP + CP * (CP + 1) / 2, NP = fwd_part_floats<CP>();
    __shared__ double delta[CP];
    const int ng = blockIdx.x, t = threadIdx.x;
    const float* mine = part + (size_t)ng * splits * NP;
    if (t < CP) {
        double s = 0.0;
        for (int q = 0; q < splits; ++q) s += (double)mine[(size_t)q * NP + t];
        delta[t] = s / hw;
        mean_in[(size_t)ng * CP + t] = (double)mine[NV + t] + s / hw;
    }
    __syncthreads();
    if (t < CP * CP) {
        const int i = t / CP, j = t % CP;
        const int k = CP + tri_index(CP, min(i, j), max(i, j));
        double s = 0.0;
        for (int q = 0; q < splits; ++q) s += (double)mine[(size_t)q * NP + k];
        cov_in[(size_t)ng * CP * CP + t] = s / hw - delta[i] * delta[j];
    }
}

// ------------------------------------------------------------------------------------------------ batch statistics

__global__ void sw_batch_mean_kernel(const double* __restrict__ mean_in, int n, int channels, double* __restrict__ mean_bn) {
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= channels) return;
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += mean_in[(size_t)i * channels + ch];
    mean_bn[ch] = s / n;
}

// grid groups, 256 threads
__global__ void __launch_bounds__(MAT_THREADS)
sw_batch_cov_kernel(const double* __restrict__ mean_in, const double* __restrict__ cov_in, const double* __restrict__ mean_bn,
                    int n, int channels, int cp, double* __restrict__ cov_bn) {
    const int g = blockIdx.x, groups = channels / cp, t = threadIdx.x;
    if (t >= cp * cp) return;
    const int i = t / cp, j = t % cp;
    const double mi = mean_bn[g * cp + i], mj = mean_bn[g * cp + j];
    double s = 0.0;
    for (int q = 0; q < n; ++q) {
        const double di = mean_in[(size_t)q * channels + g * cp + i] - mi, dj = mean_in[(size_t)q * channels + g * cp + j] - mj;
        s += cov_in[((size_t)q * groups + g) * cp * cp + t] + di * dj;
    }
    cov_bn[(size_t)g * cp * cp + t] = s / n;
}

// switchwhiten.py:101-104 in one launch, with the rounding sequence of the four torch ops:
// running = fl(fl(running * momentum) + fl((1 - momentum) * batch)), batch rounded to fp32 first.
__global__ void sw_update_running_kernel(float* __restrict__ running_mean, float* __restrict__ running_cov,
                                         const double* __restrict__ mean_bn, const double* __restrict__ cov_bn, int channels,
                                         int cov_elems, float momentum, float one_minus) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < channels)
        running_mean[t] = __fadd_rn(__fmul_rn(running_mean[t], momentum), __fmul_rn(one_minus, (float)mean_bn[t]));
    if (t < cov_elems)
        running_cov[t] = __fadd_rn(__fmul_rn(running_cov[t], momentum), __fmul_rn(one_minus, (float)cov_bn[t]));
}

// ------------------------------------------------------------------------------------------------ small matrices

// One entry of A B (optionally with transposed operands) per thread; matrices are CP x CP row-major in shared memory.
template <int CP, bool TA, bool TB>
__device__ __forceinline__ double mm(const double* a, const double* b, int i, int j) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};   // four independent chains: the fp64 pipe's latency, not its rate, is the cost
#pragma unroll
    for (int k = 0; k < CP; ++k) s[k & 3] += (TA ? a[k * CP + i] : a[i * CP + k]) * (TB ? b[j * CP + k] : b[k * CP + j]);
    return (s[0] + s[1]) + (s[2] + s[3]);
}

// What both matrix kernels share: layer statistics of the sample, the mixed mean and covariance of the
// (sample, group), and the Newton iterates P_0 .. P_T (switchwhiten.py:123-175).
template <int CP>
struct Whiten {
    double ps[MAX_T + 1][CP * CP];
    double cov[CP * CP], cov_n[CP * CP], p2[CP * CP], p3[CP * CP];
    double mean[CP];
    double red[MAT_THREADS / 32];
    double mean_ln, var_ln, r;
};

template <int CP>
__device__ void whiten_forward(Whiten<CP>& s, const Mix& m, const double* __restrict__ mean_in, const double* __restrict__ cov_in,
                               const double* __restrict__ mean_bn, const double* __restrict__ cov_bn, int ng, int channels,
                               int hw, int sw_type, int T, double eps) {
    const int groups = channels / CP, smp = ng / groups, g = ng % groups, t = threadIdx.x;
    const bool live = t < CP * CP;
    const int i = live ? t / CP : 0, j = live ? t % CP : 0;
    double mean_ln = 0.0, var_ln = 0.0;
    if (sw_type != 2) {  // switchwhiten.py:122-129, from the per-sample statistics
        const double* mi = mean_in + (size_t)smp * channels;
        const double* ci = cov_in + (size_t)smp * groups * CP * CP;
        double a = 0.0;
        for (int ch = t; ch < channels; ch += MAT_THREADS) a += mi[ch];
        mean_ln = block_sum(a, s.red) / channels;
        double q = 0.0;
        for (int ch = t; ch < channels; ch += MAT_THREADS) {
            const double d = mi[ch] - mean_ln;
            q += ci[(size_t)(ch / CP) * CP * CP + (ch % CP) * (CP + 1)] + d * d;
        }
        var_ln = block_sum(q, s.red) * ((double)hw / ((double)channels * hw - 1.0));
    }
    if (t == 0) { s.mean_ln = mean_ln; s.var_ln = var_ln; }
    if (t < CP)
        s.mean[t] = m.a_bn * mean_bn[g * CP + t] + m.a_in * mean_in[(size_t)smp * channels + g * CP + t] + m.a_ln * mean_ln;
    if (live) {
        const double cb = cov_bn[(size_t)g * CP * CP + t], ci = cov_in[(size_t)ng * CP * CP + t];
        double c = m.b_bn * cb + m.b_in * ci;
        if (i == j) c += m.d_bn * cb + m.d_in * ci + m.b_ln * var_ln + eps;
        s.cov[t] = c;
        s.ps[0][t] = i == j ? 1.0 : 0.0;
    }
    const double tr = block_sum(live && i == j ? s.cov[t] : 0.0, s.red);  // also orders the writes above
    const double r = 1.0 / tr;
    if (t == 0) s.r = r;
    if (live) s.cov_n[t] = s.cov[t] * r;
    __syncthreads();
    for (int k = 0; k < T; ++k) {   // P^3 cov_n = (P P)(P cov_n): two independent products, then one -- two barriers per iteration
        const double* p = s.ps[k];
        if (live) {
            s.p2[t] = mm<CP, false, false>(p, p, i, j);
            s.p3[t] = mm<CP, false, false>(p, s.cov_n, i, j);
        }
        __syncthreads();
        if (live) s.ps[k + 1][t] = 1.5 * p[t] - 0.5 * mm<CP, false, false>(s.p2, s.p3, i, j);
        __syncthreads();
    }
}

// grid n * groups.  a_fwd = diag(weight) wm (fp32), cst_fwd[n, ch] = bias - a_fwd mean.
template <int CP>
__global__ void __launch_bounds__(MAT_THREADS)
sw_whiten_kernel(const double* __restrict__ mean_in, const double* __restrict__ cov_in, const double* __restrict__ mean_bn,
                 const double* __restrict__ cov_bn, const float* __restrict__ mean_logits, const float* __restrict__ var_logits,
                 const float* __restrict__ weight, const float* __restrict__ bias, int channels, int hw, int sw_type, int T,
                 double eps, float* __restrict__ a_fwd, float* __restrict__ cst_fwd) {
    __shared__ Whiten<CP> s;
    const Mix m = mix_coeffs(sw_type, mean_logits, var_logits);
    const int ng = blockIdx.x, groups = channels / CP, smp = ng / groups, g = ng % groups, t = threadIdx.x;
    whiten_forward<CP>(s, m, mean_in, cov_in, mean_bn, cov_bn, ng, channels, hw, sw_type, T, eps);
    const double root = sqrt(s.r);
    if (t < CP * CP) {
        const int i = t / CP;
        const double a = (weight ? (double)weight[g * CP + i] : 1.0) * s.ps[T][t] * root;
        s.p2[t] = a;
        a_fwd[(size_t)ng * CP * CP + t] = (float)a;
    }
    __syncthreads();
    if (t < CP) {
        double c = bias ? (double)bias[g * CP + t] : 0.0;
#pragma unroll
        for (int j = 0; j < CP; ++j) c -= s.p2[t * CP + j] * s.mean[j];
        cst_fwd[(size_t)smp * channels + g * CP + t] = (float)c;
    }
}

// ------------------------------------------------------------------------------------------------ affine passes

// out[ng, i, p] = sum_j A[ng][i][j] u[ng, j, p] (+ sum_j B[ng][i][j] v[ng, j, p]) + cst[ng, i].
// grid (ceil(hw / (AFF_THREADS * AFF_PIX)), n * groups); AFF_PIX pixels per thread.
template <int CP, bool TWO, int AFF_PIX>
__global__ void __launch_bounds__(AFF_THREADS)
sw_affine_kernel(const float* __restrict__ u, const float* __restrict__ v, const float* __restrict__ a, const float* __restrict__ b,
                 const float* __restrict__ cst, int hw, float* __restrict__ out) {
    __shared__ __align__(16) float sa[CP * CP];
    __shared__ __align__(16) float sb[TWO ? CP * CP : 4];
    __shared__ float sc[CP];
    const int ng = blockIdx.y;
    for (int k = threadIdx.x; k < CP * CP; k += AFF_THREADS) {
        sa[k] = a[(size_t)ng * CP * CP + k];
        if (TWO) sb[k] = b[(size_t)ng * CP * CP + k];
    }
    if (threadIdx.x < CP) sc[threadIdx.x] = cst[(size_t)ng * CP + threadIdx.x];
    __syncthreads();
    const size_t base = (size_t)ng * CP * hw;
    const int p0 = blockIdx.x * (AFF_THREADS * AFF_PIX) + threadIdx.x;
    float in[CP][AFF_PIX], acc[CP][AFF_PIX];
#pragma unroll
    for (int j = 0; j < CP; ++j)
#pragma unroll
        for (int k = 0; k < AFF_PIX; ++k) {
            const int p = p0 + k * AFF_THREADS;
            in[j][k] = p < hw ? __ldg(u + base + (size_t)j * hw + p) : 0.f;
        }
#pragma unroll
    for (int i = 0; i < CP; ++i)
#pragma unroll
        for (int k = 0; k < AFF_PIX; ++k) acc[i][k] = sc[i];
#pragma unroll
    for (int i = 0; i < CP; ++i)
#pragma unroll
        for (int j = 0; j < CP; ++j) {
            const float c = sa[i * CP + j];
#pragma unroll
            for (int k = 0; k < AFF_PIX; ++k) acc[i][k] = fmaf(c, in[j][k], acc[i][k]);
        }
    if (TWO) {
#pragma unroll
        for (int j = 0; j < CP; ++j)
#pragma unroll
            for (int k = 0; k < AFF_PIX; ++k) {
                const int p = p0 + k * AFF_THREADS;
                in[j][k] = p < hw ? __ldg(v + base + (size_t)j * hw + p) : 0.f;
            }
#pragma unroll
        for (int i = 0; i < CP; ++i)
#pragma unroll
            for (int j = 0; j < CP; ++j) {
                const float c = sb[i * CP + j];
#pragma unroll
                for (int k = 0; k < AFF_PIX; ++k) acc[i][k] = fmaf(c, in[j][k], acc[i][k]);
            }
    }
#pragma unroll
    for (int i = 0; i < CP; ++i)
#pragma unroll
        for (int k = 0; k < AFF_PIX; ++k) {
            const int p = p0 + k * AFF_THREADS;
            if (p < hw) out[base + (size_t)i * hw + p] = acc[i][k];
        }
}

// ------------------------------------------------------------------------------------------------ moments (bwd)

// grid (splits, n * groups, CP / ROWS).  part[((ng * splits + split) * CP + row) * (CP + 1) + j]: j < CP is
// K[row][j] = sum_p gy[row, p] (x[j, p] - mean_in[j]), j == CP is s[row] = sum_p gy[row, p].
template <int CP, int ROWS>
__global__ void __launch_bounds__(MOM_THREADS, 2)
sw_backward_moments_kernel(const float* __restrict__ x, const float* __restrict__ gy, const double* __restrict__ mean_in,
                           int hw, int chunk, float* __restrict__ part) {
    constexpr int NV = ROWS * (CP + 1);
    extern __shared__ float ring_raw[];
    float (*ring)[CP + ROWS][MOM_THREADS] = reinterpret_cast<float (*)[CP + ROWS][MOM_THREADS]>(ring_raw);
    __shared__ float red[MOM_THREADS / 32][NV];
    const int ng = blockIdx.y, row0 = blockIdx.z * ROWS, tid = threadIdx.x;
    const float* xb = x + (size_t)ng * CP * hw;
    const float* gb = gy + ((size_t)ng * CP + row0) * hw;
    float centre[CP], acc[NV];
#pragma unroll
    for (int j = 0; j < CP; ++j) centre[j] = (float)mean_in[(size_t)ng * CP + j];
#pragma unroll
    for (int k = 0; k < NV; ++k) acc[k] = 0.f;
    const int p0 = blockIdx.x * chunk, p1 = min(hw, p0 + chunk);
    const int iters = ceil_div(p1 - p0, MOM_THREADS);
    auto issue = [&](int it) {
        const int p = p0 + it * MOM_THREADS + tid;
        if (it < iters && p < p1) {
#pragma unroll
            for (int j = 0; j < CP; ++j) cp_async_f32(&ring[it % BWD_STAGES][j][tid], xb + (size_t)j * hw + p);
#pragma unroll
            for (int i = 0; i < ROWS; ++i) cp_async_f32(&ring[it % BWD_STAGES][CP + i][tid], gb + (size_t)i * hw + p);
        }
        cp_async_commit();
    };
    for (int it = 0; it < BWD_STAGES - 1; ++it) issue(it);
    for (int it = 0; it < iters; ++it) {
        issue(it + BWD_STAGES - 1);
        cp_async_wait<BWD_STAGES - 1>();
        const bool valid = p0 + it * MOM_THREADS + tid < p1;
        float u[CP], w[ROWS];
#pragma unroll
        for (int j = 0; j < CP; ++j) u[j] = valid ? ring[it % BWD_STAGES][j][tid] - centre[j] : 0.f;
#pragma unroll
        for (int i = 0; i < ROWS; ++i) w[i] = valid ? ring[it % BWD_STAGES][CP + i][tid] : 0.f;
#pragma unroll
        for (int i = 0; i < ROWS; ++i) {
#pragma unroll
            for (int j = 0; j < CP; ++j) acc[i * (CP + 1) + j] = fmaf(w[i], u[j], acc[i * (CP + 1) + j]);
            acc[i * (CP + 1) + CP] += w[i];
        }
    }
    const int warp = tid >> 5, lane = tid & 31;
    float tot[(NV + 31) / 32];
    warp_transpose_sum<NV>(acc, tot);
#pragma unroll
    for (int g = 0; g < (NV + 31) / 32; ++g)
        if (g * 32 + lane < NV) red[warp][g * 32 + lane] = tot[g];
    __syncthreads();
    float* out = part + (((size_t)ng * gridDim.x + blockIdx.x) * CP + row0) * (CP + 1);
    for (int k = tid; k < NV; k += MOM_THREADS) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < MOM_THREADS / 32; ++w) s += red[w][k];
        out[k] = s;
    }
}

// ------------------------------------------------------------------------------------------------ backward matrices

struct BwdLayout {
    size_t part, g_cov, g_mean, dots, ln, gw, gb, a_fwd_cst, m1, m2, cst, total;
};

// Pixels per moments CTA: as many CTAs as one resident wave holds (2 per SM), in whole 128-pixel steps, at least
// 512 pixels so that the 150-value block reduction stays a small part of the CTA's work.
struct Split { int chunk, splits; };
__host__ inline Split plan_split(int ng, int hw, int z) {
    int want = NUM_SMS * MOM_CTAS_PER_SM / (ng * z);   // never more CTAs than one resident wave (a second, short wave costs a whole CTA time)
    const int most = ceil_div(hw, 512);
    want = want < 1 ? 1 : want > most ? most : want;
    Split s;
    s.chunk = ceil_div(ceil_div(hw, want), MOM_THREADS) * MOM_THREADS;
    s.splits = ceil_div(hw, s.chunk);
    return s;
}
__host__ inline int bwd_z(int cp) { return cp / (cp < BWD_ROWS ? cp : BWD_ROWS); }

__host__ inline BwdLayout layout(int n, int channels, int hw, int cp) {
    const size_t ng = (size_t)n * (channels / cp), mat = (size_t)cp * cp;
    const size_t fwd_part = ng * plan_split((int)ng, hw, 1).splits * (cp + cp * (cp + 1) / 2 + cp) * sizeof(float);
    const size_t bwd_part = ng * plan_split((int)ng, hw, bwd_z(cp)).splits * cp * (cp + 1) * sizeof(float);
    BwdLayout l;
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes, 256); return at; };
    l.part = take(fwd_part > bwd_part ? fwd_part : bwd_part);
    l.g_cov = take(ng * mat * sizeof(double));
    l.g_mean = take((size_t)n * channels * sizeof(double));
    l.dots = take(ng * N_DOTS * sizeof(double));
    l.ln = take((size_t)n * N_LN * sizeof(double));
    l.gw = take((size_t)n * channels * sizeof(double));
    l.gb = take((size_t)n * channels * sizeof(double));
    l.a_fwd_cst = take((size_t)n * channels * sizeof(float));
    l.m1 = take(ng * mat * sizeof(float));
    l.m2 = take(ng * mat * sizeof(float));
    l.cst = take((size_t)n * channels * sizeof(float));
    l.total = o;
    return l;
}

// grid n * groups, 256 threads.
template <int CP>
__global__ void __launch_bounds__(MAT_THREADS)
sw_backward_matrices_kernel(const float* __restrict__ part, int splits, const double* __restrict__ mean_in,
                            const double* __restrict__ cov_in, const double* __restrict__ mean_bn,
                            const double* __restrict__ cov_bn, const float* __restrict__ mean_logits,
                            const float* __restrict__ var_logits, const float* __restrict__ weight, int channels, int hw,
                            int sw_type, int T, double eps, double* __restrict__ g_cov_out, double* __restrict__ g_mean_out,
                            double* __restrict__ dots, double* __restrict__ ln, double* __restrict__ gw_part,
                            double* __restrict__ gb_part) {
    __shared__ Whiten<CP> s;
    __shared__ double gp_a[CP * CP], gp_b[CP * CP], gp3[CP * CP], tmp[CP * CP], s_gy[CP], g_mean[CP];
    const Mix m = mix_coeffs(sw_type, mean_logits, var_logits);
    const int ng = blockIdx.x, groups = channels / CP, smp = ng / groups, g = ng % groups, t = threadIdx.x;
    const bool live = t < CP * CP;
    const int i = live ? t / CP : 0, j = live ? t % CP : 0;

    // K and s from the split partials
    const float* mine = part + (size_t)ng * splits * CP * (CP + 1);
    double k_raw = 0.0;
    if (live)
        for (int q = 0; q < splits; ++q) k_raw += (double)mine[((size_t)q * CP + i) * (CP + 1) + j];
    if (t < CP) {
        double a = 0.0;
        for (int q = 0; q < splits; ++q) a += (double)mine[((size_t)q * CP + t) * (CP + 1) + CP];
        s_gy[t] = a;
    }
    whiten_forward<CP>(s, m, mean_in, cov_in, mean_bn, cov_bn, ng, channels, hw, sw_type, T, eps);  // syncs inside
    const double r = s.r, root = sqrt(r);
    const double* pt = s.ps[T];
    const size_t chan0 = (size_t)smp * channels + g * CP;

    // sum_p gy_i (x_j - mean_j), grad of weight / bias, grad of wm and of the mixed mean
    double g_wm = 0.0;
    if (live) {
        const double wi = weight ? (double)weight[g * CP + i] : 1.0;
        // the moments pass centred x on fl32(mean_in) (its registers are fp32): undo exactly that
        const double v = k_raw + s_gy[i] * ((double)(float)mean_in[chan0 + j] - s.mean[j]);
        tmp[t] = pt[t] * root * v;
        g_wm = wi * v;
    }
    __syncthreads();
    if (t < CP) {
        double a = 0.0, b = 0.0;
#pragma unroll
        for (int q = 0; q < CP; ++q) {
            a += tmp[t * CP + q];                                                              // row t of wm o Kc
            b -= pt[q * CP + t] * root * (weight ? (double)weight[g * CP + q] : 1.0) * s_gy[q];  // column t of wm
        }
        gw_part[chan0 + t] = a;
        gb_part[chan0 + t] = s_gy[t];
        g_mean[t] = b;
        g_mean_out[chan0 + t] = b;
    }
    // adjoint of wm = P_T sqrt(r), r = 1 / tr(cov), cov_n = cov r, P_{k+1} = 1.5 P_k - 0.5 P_k^3 cov_n
    double g_r = block_sum(live ? g_wm * pt[t] : 0.0, s.red) * 0.5 / root;   // (syncs: tmp / g_mean are settled)
    double g_covn = 0.0;
    double* gp = gp_a;     // G_{k+1}; the next one is written to the other buffer while this one is still being read
    double* gq = gp_b;
    if (live) gp[t] = g_wm * root;
    __syncthreads();
    // cov_n and every iterate are polynomials in the symmetric cov: they equal their transposes to fp64 rounding, so the
    // transposed right-hand operands below are read untransposed (a transposed read of a 16 x 16 fp64 matrix is a
    // 16-way shared-memory bank conflict).
    for (int k = T - 1; k >= 0; --k) {   // three barriers per iteration
        const double* p = s.ps[k];
        if (live) {
            s.p2[t] = mm<CP, false, false>(p, p, i, j);
            gp3[t] = -0.5 * mm<CP, false, false>(gp, s.cov_n, i, j);          // cov_n^T = cov_n
        }
        __syncthreads();
        double next = 0.0;
        if (live) {
            s.p3[t] = mm<CP, false, false>(s.p2, p, i, j);
            tmp[t] = mm<CP, true, false>(p, gp3, i, j);                       // P^T G3
            next = 1.5 * gp[t] + mm<CP, false, false>(gp3, s.p2, i, j) + mm<CP, true, false>(s.p2, gp3, i, j);
        }
        __syncthreads();
        if (live) {
            g_covn += -0.5 * mm<CP, true, false>(s.p3, gp, i, j);
            gq[t] = next + mm<CP, false, false>(tmp, p, i, j);                 // + P^T G3 P^T
        }
        __syncthreads();
        double* swap = gp; gp = gq; gq = swap;
    }
    g_r += block_sum(live ? g_covn * s.cov[t] : 0.0, s.red);
    double g_cov = 0.0;
    if (live) {
        g_cov = g_covn * r + (i == j ? -g_r * r * r : 0.0);
        g_cov_out[(size_t)ng * CP * CP + t] = g_cov;
    }

    // the dot products the weight gradients and the layer-statistics adjoints are made of
    const double cb = live ? cov_bn[(size_t)g * CP * CP + t] : 0.0, ci = live ? cov_in[(size_t)ng * CP * CP + t] : 0.0;
    const bool diag = live && i == j;
    double d[N_DOTS];
    d[D_COV_BN] = block_sum(g_cov * cb, s.red);
    d[D_COV_IN] = block_sum(g_cov * ci, s.red);
    d[D_DIAG_BN] = block_sum(diag ? g_cov * cb : 0.0, s.red);
    d[D_DIAG_IN] = block_sum(diag ? g_cov * ci : 0.0, s.red);
    d[D_TR] = block_sum(diag ? g_cov : 0.0, s.red);
    d[D_TR_VARLN] = d[D_TR] * s.var_ln;
    d[D_MEAN_BN] = block_sum(t < CP ? g_mean[t] * mean_bn[g * CP + t] : 0.0, s.red);
    d[D_MEAN_IN] = block_sum(t < CP ? g_mean[t] * mean_in[chan0 + t] : 0.0, s.red);
    d[D_SUM_GMEAN] = block_sum(t < CP ? g_mean[t] : 0.0, s.red);
    d[D_GMEAN_MEANLN] = d[D_SUM_GMEAN] * s.mean_ln;
    if (t == 0) {
#pragma unroll
        for (int q = 0; q < N_DOTS; ++q) dots[(size_t)ng * N_DOTS + q] = d[q];
        if (g == 0) { ln[(size_t)smp * N_LN + L_MEAN] = s.mean_ln; ln[(size_t)smp * N_LN + L_VAR] = s.var_ln; }
    }
}

// Reductions over samples / groups.  grid max(groups, n) + 1, 256 threads:
//   block b < groups : adjoints of the batch statistics of group b, grad of weight / bias of its channels
//   block b < n      : adjoints of the layer statistics of sample b
//   last block       : gradients of the two importance-weight vectors (switchwhiten.py:137-164, softmax backward)
__global__ void __launch_bounds__(MAT_THREADS)
sw_backward_reduce_kernel(const double* __restrict__ g_cov, const double* __restrict__ g_mean, const double* __restrict__ dots,
                          const double* __restrict__ gw_part, const double* __restrict__ gb_part,
                          const float* __restrict__ mean_logits, const float* __restrict__ var_logits, int n, int channels,
                          int cp, int sw_type, double* __restrict__ ln, double* __restrict__ g_mean_bn,
                          double* __restrict__ g_cov_bn, float* __restrict__ g_weight, float* __restrict__ g_bias,
                          float* __restrict__ g_sw_mean, float* __restrict__ g_sw_var) {
    __shared__ double red[MAT_THREADS / 32];
    const Mix m = mix_coeffs(sw_type, mean_logits, var_logits);
    const int groups = channels / cp, b = blockIdx.x, t = threadIdx.x;
    if (b < groups) {
        if (t < cp * cp) {
            const int i = t / cp, j = t % cp;
            double s = 0.0;
            for (int q = 0; q < n; ++q) s += g_cov[((size_t)q * groups + b) * cp * cp + t];
            g_cov_bn[(size_t)b * cp * cp + t] = (i == j ? m.b_bn + m.d_bn : m.b_bn) * s;
        }
        if (t < cp) {
            const int ch = b * cp + t;
            double s = 0.0, w = 0.0, c = 0.0;
            for (int q = 0; q < n; ++q) {
                s += g_mean[(size_t)q * channels + ch];
                w += gw_part[(size_t)q * channels + ch];
                c += gb_part[(size_t)q * channels + ch];
            }
            g_mean_bn[ch] = m.a_bn * s;
            if (g_weight) g_weight[ch] = (float)w;
            if (g_bias) g_bias[ch] = (float)c;
        }
    }
    if (b < n && t == 0) {
        double tr = 0.0, sm = 0.0;
        for (int g = 0; g < groups; ++g) {
            tr += dots[((size_t)b * groups + g) * N_DOTS + D_TR];
            sm += dots[((size_t)b * groups + g) * N_DOTS + D_SUM_GMEAN];
        }
        ln[(size_t)b * N_LN + L_G_VAR] = m.b_ln * tr;
        ln[(size_t)b * N_LN + L_G_MEAN] = m.a_ln * sm;
    }
    if (b == (int)gridDim.x - 1) {
        double d[N_DOTS];
        for (int q = 0; q < N_DOTS; ++q) {
            double a = 0.0;
            for (int k = t; k < n * groups; k += MAT_THREADS) a += dots[(size_t)k * N_DOTS + q];
            d[q] = block_sum(a, red);
        }
        if (t == 0) {
            double gm[5] = {0, 0, 0, 0, 0}, gv[5] = {0, 0, 0, 0, 0};
            gm[0] = d[D_MEAN_BN]; gm[1] = d[D_MEAN_IN];
            gv[0] = d[D_COV_BN]; gv[1] = d[D_COV_IN];
            if (sw_type == 3) { gm[2] = d[D_GMEAN_MEANLN]; gv[2] = d[D_TR_VARLN]; }
            if (sw_type == 5) {
                gm[2] = d[D_MEAN_BN]; gm[3] = d[D_MEAN_IN]; gm[4] = d[D_GMEAN_MEANLN];
                gv[0] += d[D_DIAG_BN]; gv[1] += d[D_DIAG_IN]; gv[4] = d[D_TR_VARLN];
            }
            if (!g_sw_var)  // tie_weight: one vector feeds both mixes
                for (int q = 0; q < sw_type; ++q) gm[q] += gv[q];
            double dm = 0.0, dv = 0.0;
            for (int q = 0; q < sw_type; ++q) { dm += m.mw[q] * gm[q]; dv += m.vw[q] * gv[q]; }
            for (int q = 0; q < sw_type; ++q) {
                g_sw_mean[q] = (float)(m.mw[q] * (gm[q] - dm));
                if (g_sw_var) g_sw_var[q] = (float)(m.vw[q] * (gv[q] - dv));
            }
        }
    }
}

// grid n * groups, 256 threads: M1 = a_fwd^T, M2 = S_in + S_bn, cst (oracle: "backward affine pass").
template <int CP>
__global__ void __launch_bounds__(MAT_THREADS)
sw_backward_coeffs_kernel(const float* __restrict__ a_fwd, const double* __restrict__ g_cov, const double* __restrict__ g_mean,
                          const double* __restrict__ ln, const double* __restrict__ mean_in, const double* __restrict__ mean_bn,
                          const double* __restrict__ g_mean_bn, const double* __restrict__ g_cov_bn,
                          const float* __restrict__ mean_logits, const float* __restrict__ var_logits, double bn_scale,
                          int channels, int hw, int sw_type, float* __restrict__ m1, float* __restrict__ m2,
                          float* __restrict__ cst) {
    __shared__ double sin_[CP * CP], sbn[CP * CP];
    const Mix m = mix_coeffs(sw_type, mean_logits, var_logits);
    const int ng = blockIdx.x, groups = channels / CP, smp = ng / groups, g = ng % groups, t = threadIdx.x;
    const double ln_scale = (double)hw / ((double)channels * hw - 1.0);
    const double g_var_ln = sw_type == 2 ? 0.0 : ln[(size_t)smp * N_LN + L_G_VAR];
    const double g_mean_ln = sw_type == 2 ? 0.0 : ln[(size_t)smp * N_LN + L_G_MEAN];
    const double mean_ln = sw_type == 2 ? 0.0 : ln[(size_t)smp * N_LN + L_MEAN];
    if (t < CP * CP) {
        const int i = t / CP, j = t % CP, tt = j * CP + i;
        const double* gc = g_cov + (size_t)ng * CP * CP;
        double a = m.b_in * (gc[t] + gc[tt]);
        if (i == j) a += 2.0 * (m.d_in * gc[t] + g_var_ln * ln_scale);
        a /= hw;
        const double* gb = g_cov_bn + (size_t)g * CP * CP;
        const double c = (gb[t] + gb[tt]) * bn_scale;
        sin_[t] = a;
        sbn[t] = c;
        m1[(size_t)ng * CP * CP + t] = a_fwd[(size_t)ng * CP * CP + tt];
        m2[(size_t)ng * CP * CP + t] = (float)(a + c);
    }
    __syncthreads();
    if (t < CP) {
        const size_t ch = (size_t)smp * channels + g * CP + t;
        const double g_mean_in = m.a_in * g_mean[ch] + g_mean_ln / channels +
                                 g_var_ln * ln_scale * 2.0 * (mean_in[ch] - mean_ln);
        double c = g_mean_in / hw + g_mean_bn[g * CP + t] * bn_scale;
#pragma unroll
        for (int j = 0; j < CP; ++j)
            c -= sin_[t * CP + j] * mean_in[(size_t)smp * channels + g * CP + j] + sbn[t * CP + j] * mean_bn[g * CP + j];
        cst[ch] = (float)c;
    }
}

// ------------------------------------------------------------------------------------------------ host side

inline bool bad_shape(int n, int channels, int hw, int cp) {
    return n <= 0 || channels <= 0 || hw <= 0 || (cp != 4 && cp != 8 && cp != 16) || channels % cp != 0;
}
inline bool bad_mix(int sw_type, int T) { return (sw_type != 2 && sw_type != 3 && sw_type != 5) || T < 1 || T > MAX_T; }

#define SW_DISPATCH(cp, CALL)                  \
    do {                                       \
        if ((cp) == 16) { CALL(16); }          \
        else if ((cp) == 8) { CALL(8); }       \
        else { CALL(4); }                      \
    } while (0)

template <int CP, bool TWO>
void launch_affine(const float* u, const float* v, const float* a, const float* b, const float* cst, int ng, int hw,
                   float* out, cudaStream_t st) {
    // 4 pixels per thread: 168 registers, 3 CTAs per SM; 2 pixels (128 registers, 4 CTAs) measured 10 % slower
    sw_affine_kernel<CP, TWO, 4><<<dim3(ceil_div(hw, AFF_THREADS * 4), ng), AFF_THREADS, 0, st>>>(u, v, a, b, cst, hw, out);
}

template <int CP>
cudaError_t launch_moments(const float* x, int ng, int hw, Split sp, float* part, cudaStream_t st) {
    constexpr int SMEM = FWD_STAGES * CP * MOM_THREADS * (int)sizeof(float);
    static bool configured[MAX_DEVICES] = {};   // the attribute is per device
    int device = 0;
    if (cudaGetDevice(&device) != cudaSuccess || device < 0 || device >= MAX_DEVICES) return cudaErrorInvalidDevice;
    if (!configured[device]) {
        const cudaError_t e = cudaFuncSetAttribute(sw_moments_kernel<CP>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e != cudaSuccess) return e;
        configured[device] = true;
    }
    sw_moments_kernel<CP><<<dim3(sp.splits, ng), MOM_THREADS, SMEM, st>>>(x, hw, sp.chunk, part);
    return cudaSuccess;
}

template <int CP>
cudaError_t launch_backward_moments(const float* x, const float* gy, const double* mean_in, int ng, int hw, Split sp,
                                    float* part, cudaStream_t st) {
    constexpr int ROWS = CP < BWD_ROWS ? CP : BWD_ROWS;
    constexpr int SMEM = BWD_STAGES * (CP + ROWS) * MOM_THREADS * (int)sizeof(float);
    static bool configured[MAX_DEVICES] = {};
    int device = 0;
    if (cudaGetDevice(&device) != cudaSuccess || device < 0 || device >= MAX_DEVICES) return cudaErrorInvalidDevice;
    if (!configured[device]) {
        const cudaError_t e = cudaFuncSetAttribute(sw_backward_moments_kernel<CP, ROWS>,
                                                   cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e != cudaSuccess) return e;
        configured[device] = true;
    }
    sw_backward_moments_kernel<CP, ROWS><<<dim3(sp.splits, ng, CP / ROWS), MOM_THREADS, SMEM, st>>>(x, gy, mean_in, hw,
                                                                                                  sp.chunk, part);
    return cudaSuccess;
}

}  // namespace sw
}  // namespace dgvcc

using namespace dgvcc;
using namespace dgvcc::sw;

extern "C" size_t dgvcc_sw_workspace_bytes(int n, int channels, int hw, int num_pergroup) {
    if (bad_shape(n, channels, hw, num_pergroup)) return 0;
    return layout(n, channels, hw, num_pergroup).total;
}

extern "C" int dgvcc_sw_instance_stats(const float* x, int n, int channels, int hw, int num_pergroup, double* mean_in,
                                       double* cov_in, void* workspace, size_t workspace_bytes, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !mean_in || !cov_in || !workspace || bad_shape(n, channels, hw, num_pergroup)) return DGVCC_ERR_ARG;
    const BwdLayout l = layout(n, channels, hw, num_pergroup);
    if (workspace_bytes < l.total) return DGVCC_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int ng = n * (channels / num_pergroup);
    const Split sp = plan_split(ng, hw, 1);
    float* part = (float*)((char*)workspace + l.part);
#define CALL(CP)                                                                                             \
    DGVCC_RETURN_IF_CUDA(launch_moments<CP>(x, ng, hw, sp, part, st));                                       \
    sw_instance_stats_kernel<CP><<<ng, MAT_THREADS, 0, st>>>(part, sp.splits, hw, mean_in, cov_in)
    SW_DISPATCH(num_pergroup, CALL);
#undef CALL
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return DGVCC_OK;
}

extern "C" int dgvcc_sw_batch_mean(const double* mean_in, int n, int channels, double* mean_bn, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!mean_in || !mean_bn || n <= 0 || channels <= 0) return DGVCC_ERR_ARG;
    sw_batch_mean_kernel<<<ceil_div(channels, 128), 128, 0, (cudaStream_t)stream>>>(mean_in, n, channels, mean_bn);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return DGVCC_OK;
}

extern "C" int dgvcc_sw_batch_cov(const double* mean_in, const double* cov_in, const double* mean_bn, int n, int channels,
                                  int num_pergroup, double* cov_bn, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!mean_in || !cov_in || !mean_bn || !cov_bn || bad_shape(n, channels, 1, num_pergroup)) return DGVCC_ERR_ARG;
    sw_batch_cov_kernel<<<channels / num_pergroup, MAT_THREADS, 0, (cudaStream_t)stream>>>(mean_in, cov_in, mean_bn, n,
                                                                                         channels, num_pergroup, cov_bn);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return DGVCC_OK;
}

extern "C" int dgvcc_sw_update_running(float* running_mean, float* running_cov, const double* mean_bn,
                                       const double* cov_bn, int channels, int num_pergroup, double momentum,
                                       double one_minus_momentum, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!running_mean || !running_cov || !mean_bn || !cov_bn || bad_shape(1, channels, 1, num_pergroup)) return DGVCC_ERR_ARG;
    const int cov_elems = channels * num_pergroup;
    sw_update_running_kernel<<<ceil_div(cov_elems, 256), 256, 0, (cudaStream_t)stream>>>(
        running_mean, running_cov, mean_bn, cov_bn, channels, cov_elems, (float)momentum, (float)one_minus_momentum);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return DGVCC_OK;
}

extern "C" int dgvcc_sw_whiten_forward(const float* x, const double* mean_in, const double* cov_in, const double* mean_bn,
                                       const double* cov_bn, const float* sw_mean_weight, const float* sw_var_weight,
                                       const float* weight, const float* bias, int n, int channels, int hw,
                                       int num_pergroup, int sw_type, int T, float eps, float* a_fwd, float* y,
                                       void* workspace, size_t workspace_bytes, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !mean_in || !cov_in || !mean_bn || !cov_bn || !sw_mean_weight || !a_fwd || !y || !workspace ||
        (weight == nullptr) != (bias == nullptr) || bad_shape(n, channels, hw, num_pergroup) || bad_mix(sw_type, T))
        return DGVCC_ERR_ARG;
    const BwdLayout l = layout(n, channels, hw, num_pergroup);
    if (workspace_bytes < l.total) return DGVCC_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int ng = n * (channels / num_pergroup);
    float* cst = (float*)((char*)workspace + l.a_fwd_cst);
#define CALL(CP)                                                                                                      \
    sw_whiten_kernel<CP><<<ng, MAT_THREADS, 0, st>>>(mean_in, cov_in, mean_bn, cov_bn, sw_mean_weight, sw_var_weight,   \
                                                    weight, bias, channels, hw, sw_type, T, (double)eps, a_fwd, cst);  \
    launch_affine<CP, false>(x, nullptr, a_fwd, nullptr, cst, ng, hw, y, st)
    SW_DISPATCH(num_pergroup, CALL);
#undef CALL
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return DGVCC_OK;
}

extern "C" int dgvcc_sw_backward_stats(const float* x, const float* grad_y, const double* mean_in, const double* cov_in,
                                       const double* mean_bn, const double* cov_bn, const float* sw_mean_weight,
                                       const float* sw_var_weight, const float* weight, int n, int channels, int hw,
                                       int num_pergroup, int sw_type, int T, float eps, float* grad_sw_mean,
                                       float* grad_sw_var, float* grad_weight, float* grad_bias, double* grad_mean_bn,
                                       double* grad_cov_bn, void* workspace, size_t workspace_bytes, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !grad_y || !mean_in || !cov_in || !mean_bn || !cov_bn || !sw_mean_weight || !grad_sw_mean || !grad_mean_bn ||
        !grad_cov_bn || !workspace || (sw_var_weight == nullptr) != (grad_sw_var == nullptr) ||
        bad_shape(n, channels, hw, num_pergroup) || bad_mix(sw_type, T))
        return DGVCC_ERR_ARG;
    const BwdLayout l = layout(n, channels, hw, num_pergroup);
    if (workspace_bytes < l.total) return DGVCC_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int groups = channels / num_pergroup, ng = n * groups;
    const Split sp = plan_split(ng, hw, bwd_z(num_pergroup));
    const int splits = sp.splits;
    char* ws = (char*)workspace;
    float* part = (float*)(ws + l.part);
    double *g_cov = (double*)(ws + l.g_cov), *g_mean = (double*)(ws + l.g_mean), *dots = (double*)(ws + l.dots),
           *ln = (double*)(ws + l.ln), *gw = (double*)(ws + l.gw), *gb = (double*)(ws + l.gb);
#define CALL(CP)                                                                                                      \
    DGVCC_RETURN_IF_CUDA(launch_backward_moments<CP>(x, grad_y, mean_in, ng, hw, sp, part, st));                                              \
    sw_backward_matrices_kernel<CP><<<ng, MAT_THREADS, 0, st>>>(part, splits, mean_in, cov_in, mean_bn, cov_bn,        \
                                                               sw_mean_weight, sw_var_weight, weight, channels, hw,   \
                                                               sw_type, T, (double)eps, g_cov, g_mean, dots, ln, gw, gb)
    SW_DISPATCH(num_pergroup, CALL);
#undef CALL
    const int blocks = (groups > n ? groups : n) + 1;
    sw_backward_reduce_kernel<<<blocks, MAT_THREADS, 0, st>>>(g_cov, g_mean, dots, gw, gb, sw_mean_weight, sw_var_weight, n,
                                                             channels, num_pergroup, sw_type, ln, grad_mean_bn, grad_cov_bn,
                                                             grad_weight, grad_bias, grad_sw_mean, grad_sw_var);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return DGVCC_OK;
}

extern "C" int dgvcc_sw_backward_apply(const float* x, const float* grad_y, const float* a_fwd, const double* mean_in,
                                       const double* mean_bn, const double* grad_mean_bn, const double* grad_cov_bn,
                                       const float* sw_mean_weight, const float* sw_var_weight, double bn_scale, int n,
                                       int channels, int hw, int num_pergroup, int sw_type, float* grad_x,
                                       void* workspace, size_t workspace_bytes, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !grad_y || !a_fwd || !mean_in || !mean_bn || !grad_mean_bn || !grad_cov_bn || !sw_mean_weight || !grad_x ||
        !workspace || bad_shape(n, channels, hw, num_pergroup) || bad_mix(sw_type, 1))
        return DGVCC_ERR_ARG;
    const BwdLayout l = layout(n, channels, hw, num_pergroup);
    if (workspace_bytes < l.total) return DGVCC_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int ng = n * (channels / num_pergroup);
    char* ws = (char*)workspace;
    float *m1 = (float*)(ws + l.m1), *m2 = (float*)(ws + l.m2), *cst = (float*)(ws + l.cst);
#define CALL(CP)                                                                                                      \
    sw_backward_coeffs_kernel<CP><<<ng, MAT_THREADS, 0, st>>>(a_fwd, (const double*)(ws + l.g_cov),                   \
                                                             (const double*)(ws + l.g_mean), (const double*)(ws + l.ln), \
                                                             mean_in, mean_bn, grad_mean_bn, grad_cov_bn, sw_mean_weight, \
                                                             sw_var_weight, bn_scale, channels, hw, sw_type, m1, m2, cst); \
    launch_affine<CP, true>(grad_y, x, m1, m2, cst, ng, hw, grad_x, st)
    SW_DISPATCH(num_pergroup, CALL);
#undef CALL
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return DGVCC_OK;
}
