// ISW instance-whitening covariance loss for sm_100a: everything around the Gram contraction.
//
// Replaces models/ISW/instance_whitening.py of the reference:
//   isw_instnorm_fwd/bwd_kernel : nn.InstanceNorm2d(dim, affine=False)            instance_whitening.py:5-16
//   isw_gram_simt_kernel        : exact-fp32 split-K Gram partials X X^T (CUDA cores); used for channel
//                                 counts the tensor-core kernel (isw_gram_tc.cu) does not tile, and as its
//                                 cross-check in the tests                        instance_whitening.py:37
//   isw_cov_finish_kernel       : fixed-order sum of the split-K partials, /(HW-1) + eps*eye, mirrored to
//                                 the full symmetric [C,C]                        instance_whitening.py:37
//   isw_loss_kernel             : sum |f_cor*mask| - margin, /num_remove_cov, clamp, mean over B
//                                                                                 instance_whitening.py:19-27
//   isw_loss_grad_kernel        : S_b = dL/df_cor_b symmetrised / (HW-1)          autograd of :19-39
//   isw_sx_simt_kernel          : dX_b = S_b X_b  (exact fp32; the tensor-core version is isw_sx_tc.cu)
//                                                                                 autograd of :37
// Deterministic: no float atomics; split-K partials are added in split order.
// Half-precision feature maps (fp16 / bf16, the *_h entry points): the instance norm is templated over the element type
// and the Gram / dX = S X run the half variants of the tensor-core kernels; every value is the one the fp32 path computes
// on the upcast map (DESIGN section 5).
#include <type_traits>

#include "isw_tc.cuh"
#include "tc_common.cuh"
#include "../../include/dgvcc_b200.h"

namespace dgvcc {
namespace isw {

// ------------------------------------------------------------------------------- instance norm
constexpr int NORM_THREADS = 256;

__device__ __forceinline__ float block_sum(float v, float* scratch) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < NORM_THREADS / 32; ++w) t += scratch[w];
    return t;  // same value on every thread, fixed order
}

// Element access of the instance norm: fp32 as it is, fp16 / bf16 widened exactly on load and rounded to nearest on store.
template <typename T> struct Elem {
    static __device__ __forceinline__ float load(T v) { return dgvcc::tc::HalfIn<T>::widen(v); }
    static __device__ __forceinline__ T store(float v) { return dgvcc::tc::HalfIn<T>::narrow(v); }
};
template <> struct Elem<float> {
    static __device__ __forceinline__ float load(float v) { return v; }
    static __device__ __forceinline__ float store(float v) { return v; }
};

// One CTA per (b, c) plane of HW elements: mean, biased variance (two-pass on the cached plane), normalise.
// T = __half / __nv_bfloat16: the plane is cached in the input type (twice the plane fits) and y is written as RN(y).
template <typename T>
__global__ void __launch_bounds__(NORM_THREADS)
isw_instnorm_fwd_kernel(const T* __restrict__ x, int hw, float eps, T* __restrict__ y,
                        float* __restrict__ mean_out, float* __restrict__ invstd_out) {
    extern __shared__ float plane_f32[];  // hw elements when they fit, else unused
    T* plane = reinterpret_cast<T*>(plane_f32);
    __shared__ float scratch[NORM_THREADS / 32];
    const size_t base = (size_t)blockIdx.x * hw;
    const bool cached = gridDim.y == 1;  // launch with gridDim.y == 2 to signal "does not fit in smem"
    const T* src = x + base;
    float s = 0.f;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const T v = src[i];
        if (cached) plane[i] = v;
        s += Elem<T>::load(v);
    }
    const float mean = block_sum(s, scratch) / (float)hw;
    float q = 0.f;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float d = Elem<T>::load(cached ? plane[i] : src[i]) - mean;
        q = fmaf(d, d, q);
    }
    const float var = block_sum(q, scratch) / (float)hw;
    const float invstd = 1.0f / sqrtf(var + eps);
    if (blockIdx.y == 0) {
        for (int i = threadIdx.x; i < hw; i += NORM_THREADS)
            y[base + i] = Elem<T>::store((Elem<T>::load(cached ? plane[i] : src[i]) - mean) * invstd);
        if (threadIdx.x == 0) { mean_out[blockIdx.x] = mean; invstd_out[blockIdx.x] = invstd; }
    }
}

// dx = invstd * (dy - mean(dy) - y * mean(dy * y))
__global__ void __launch_bounds__(NORM_THREADS)
isw_instnorm_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y, const float* __restrict__ invstd,
                        int hw, float* __restrict__ dx) {
    __shared__ float scratch[NORM_THREADS / 32];
    const size_t base = (size_t)blockIdx.x * hw;
    float s1 = 0.f, s2 = 0.f;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float g = dy[base + i];
        s1 += g;
        s2 = fmaf(g, y[base + i], s2);
    }
    const float m1 = block_sum(s1, scratch) / (float)hw;
    const float m2 = block_sum(s2, scratch) / (float)hw;
    const float is = invstd[blockIdx.x];
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS)
        dx[base + i] = is * (dy[base + i] - m1 - y[base + i] * m2);
}

// The same for a half-precision plane, from x, mean and invstd instead of a saved fp32 y: y is recomputed with the
// forward's operations ((v - mean) * invstd: a sub and a mul, nothing to contract), so it is the forward's fp32 y bit for
// bit; dx is written as RN(dx).
template <typename T>
__global__ void __launch_bounds__(NORM_THREADS)
isw_instnorm_bwd_half_kernel(const T* __restrict__ dy, const T* __restrict__ x, const float* __restrict__ mean,
                             const float* __restrict__ invstd, int hw, T* __restrict__ dx) {
    __shared__ float scratch[NORM_THREADS / 32];
    const size_t base = (size_t)blockIdx.x * hw;
    const float mu = mean[blockIdx.x], is = invstd[blockIdx.x];
    float s1 = 0.f, s2 = 0.f;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float g = Elem<T>::load(dy[base + i]);
        s1 += g;
        s2 = fmaf(g, __fmul_rn(__fsub_rn(Elem<T>::load(x[base + i]), mu), is), s2);
    }
    const float m1 = block_sum(s1, scratch) / (float)hw;
    const float m2 = block_sum(s2, scratch) / (float)hw;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float yv = __fmul_rn(__fsub_rn(Elem<T>::load(x[base + i]), mu), is);
        dx[base + i] = Elem<T>::store(is * (Elem<T>::load(dy[base + i]) - m1 - yv * m2));
    }
}

// ------------------------------------------------------------------------------- SIMT Gram
constexpr int GT = 64;        // output tile edge
constexpr int GK = 16;        // k-chunk
constexpr int GEMM_THREADS = 256;

// part[((b*splits + split)*n_tiles + tile)][64][64] = X_I X_J^T over this split's k-range, tiles J >= I.
__global__ void __launch_bounds__(GEMM_THREADS)
isw_gram_simt_kernel(const float* __restrict__ x, int c, int hw, int splits, int k_per_split,
                     float* __restrict__ part) {
    __shared__ float as[GK][GT + 4];
    __shared__ float bs[GK][GT + 4];
    const int tiles_1d = (c + GT - 1) / GT;
    // upper-triangular tile index -> (ti, tj), tj >= ti
    int ti = 0, rem = blockIdx.x;
    while (rem >= tiles_1d - ti) { rem -= tiles_1d - ti; ++ti; }
    const int tj = ti + rem;
    const int split = blockIdx.y, b = blockIdx.z;
    const int k0 = split * k_per_split, k1 = min(hw, k0 + k_per_split);
    const float* xb = x + (size_t)b * c * hw;
    const int tid = threadIdx.x;
    const int lr = tid >> 2, lk = (tid & 3) * 4;  // loader: row lr of the tile, 4 consecutive k
    const int ty = tid >> 4, tx = tid & 15;        // compute: 4x4 outputs at rows ty*4.., cols tx*4..
    float acc[4][4] = {};
    for (int kb = k0; kb < k1; kb += GK) {
        float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
        const int ra = ti * GT + lr, rb = tj * GT + lr;
        float* pa = reinterpret_cast<float*>(&va);
        float* pb = reinterpret_cast<float*>(&vb);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int k = kb + lk + q;
            if (k < k1) {
                if (ra < c) pa[q] = xb[(size_t)ra * hw + k];
                if (rb < c) pb[q] = xb[(size_t)rb * hw + k];
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) { as[lk + q][lr] = pa[q]; bs[lk + q][lr] = pb[q]; }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < GK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&as[k][ty * 4]);
            const float4 bb = *reinterpret_cast<const float4*>(&bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
    }
    const int n_tiles = tiles_1d * (tiles_1d + 1) / 2;
    float* out = part + (((size_t)b * splits + split) * n_tiles + blockIdx.x) * GT * GT;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(&out[(ty * 4 + i) * GT + tx * 4]) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
}

// f_cor[b][i][j] = sum_split part / (hw-1) + eps*eye[i][j], written to both (i,j) and (j,i).
// `tile` is the edge of the partial tiles (64 for the SIMT kernel, 128 for the tensor-core kernel).
// One CTA (32 x 8 threads) owns a 32 x 32 block of a partial tile: it adds the splits in order (coalesced rows),
// stores the block, and stores its mirror image through a shared-memory transpose, so both stores are coalesced.
// One writer per entry: on diagonal tiles the upper triangle is what gets mirrored.
__global__ void __launch_bounds__(256)
isw_cov_finish_kernel(const float* __restrict__ part, int c, float denom, int splits, int tile, const float* __restrict__ eye,
                      float eps, float* __restrict__ f_cor) {
    __shared__ float tr[32][33];
    const int tiles_1d = (c + tile - 1) / tile;
    const int n_tiles = tiles_1d * (tiles_1d + 1) / 2;
    int ti = 0, rem = blockIdx.x;
    while (rem >= tiles_1d - ti) { rem -= tiles_1d - ti; ++ti; }
    const int tj = ti + rem;
    const int b = blockIdx.z;
    const int sub = tile / 32, sy = blockIdx.y / sub, sx = blockIdx.y % sub;
    if (ti == tj && sx < sy) return;  // below the diagonal of a diagonal tile: written by the mirror of (sx, sy)
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const size_t tile_elems = (size_t)tile * tile;
    const float* p0 = part + ((size_t)b * splits * n_tiles + blockIdx.x) * tile_elems;
    float* fc = f_cor + (size_t)b * c * c;
    const int i0 = ti * tile + 32 * sy, j0 = tj * tile + 32 * sx;
    const bool diag_block = ti == tj && sx == sy;
    // denom = HW - 1 for the covariance (instance_whitening.py:37), 1 for a raw Gram; eye == NULL: no eps * eye term
    // the thread's four rows are summed side by side (independent chains, loads of several splits in flight);
    // each entry still adds its splits in split order
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    const float* p = p0 + (size_t)(32 * sy + ty) * tile + 32 * sx + tx;
    const size_t split_stride = (size_t)n_tiles * tile_elems;
#pragma unroll 4
    for (int sp = 0; sp < splits; ++sp) {
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[r] += p[(size_t)sp * split_stride + (size_t)(8 * r) * tile];
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int li = ty + 8 * r, i = i0 + li, j = j0 + tx;
        // torch: bmm(...).div(HW-1) is a true division; + (eps * eye)
        const float v = acc[r] / denom;
        tr[li][tx] = v;
        if (i < c && j < c && (!diag_block || tx >= li)) fc[(size_t)i * c + j] = eye ? v + eps * eye[(size_t)i * c + j] : v;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int lj = ty + 8 * r, j = j0 + lj, i = i0 + tx;  // entry (j, i) = mirror of (i, j) = tr[tx][lj]
        if (i < c && j < c && (!diag_block || lj > tx))
            fc[(size_t)j * c + i] = eye ? tr[tx][lj] + eps * eye[(size_t)j * c + i] : tr[tx][lj];
    }
}

// ------------------------------------------------------------------------------- loss
// off[b] = sum_ij |f_cor[b,i,j] * mask[i,j]| - margin; loss = sum_b max(off[b] / num_remove, 0) / B.
// Each sample is cut into up to LOSS_CHUNKS slices (one CTA each, fixed-order block sums); the last CTA to
// finish adds the slices of every sample in slice order and then the samples in order: deterministic, no
// float atomics.  off_out holds off[B] followed by the [B][LOSS_CHUNKS] partial sums.
constexpr int LOSS_CHUNKS = 32;

__global__ void __launch_bounds__(256)
isw_loss_kernel(const float* __restrict__ f_cor, const float* __restrict__ mask, int c, int batch,
                const float* __restrict__ margin, const float* __restrict__ num_remove, float* __restrict__ off_out,
                float* __restrict__ loss_out, unsigned int* __restrict__ ticket) {
    __shared__ float scratch[8];
    __shared__ bool s_last;
    const int b = blockIdx.y, chunks = gridDim.x;
    const int cc = c * c;
    const int per = ceil_div(ceil_div(cc, chunks), 4) * 4;  // float4-aligned slices (cc is a multiple of 4 or handled below)
    const int e0 = blockIdx.x * per, e1 = min(cc, e0 + per);
    const float* fc = f_cor + (size_t)b * cc;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if ((cc & 3) == 0 && (((uintptr_t)fc | (uintptr_t)mask) & 15u) == 0) {
        for (int e = e0 + 4 * threadIdx.x; e < e1; e += 4 * 256) {
            const float4 f = *reinterpret_cast<const float4*>(fc + e);
            const float4 m = *reinterpret_cast<const float4*>(mask + e);
            s0 += fabsf(f.x * m.x); s1 += fabsf(f.y * m.y); s2 += fabsf(f.z * m.z); s3 += fabsf(f.w * m.w);
        }
    } else {
        for (int e = e0 + threadIdx.x; e < e1; e += 256) s0 += fabsf(fc[e] * mask[e]);
    }
    float s = warp_sum((s0 + s1) + (s2 + s3));
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += scratch[w];
        float* part = off_out + batch;
        part[b * LOSS_CHUNKS + blockIdx.x] = t;
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == (unsigned)(batch * chunks) - 1u;
    }
    __syncthreads();
    if (!s_last) return;
    // last CTA: one thread per sample adds its slices in slice order, thread 0 then adds the samples in order
    __threadfence();
    const volatile float* pv = off_out + batch;
    for (int i = threadIdx.x; i < batch; i += 256) {
        float o = 0.f;
        for (int k = 0; k < chunks; ++k) o += pv[i * LOSS_CHUNKS + k];
        off_out[i] = o - margin[0];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float total = 0.f;
        for (int i = 0; i < batch; ++i) total += fmaxf(off_out[i] / num_remove[0], 0.f);
        loss_out[0] = total / (float)batch;
        *ticket = 0u;
    }
}

// S_b[i][j] = g * gate_b * (sgn(fc_ij * m_ij) * m_ij + sgn(fc_ji * m_ji) * m_ji) / (num_remove * B * (hw-1))
// with gate_b = [off_b / num_remove >= 0]  (torch clamp passes the gradient at the boundary).
// One CTA (32 x 8 threads) per 32 x 32 block: the (j,i) terms come from the mirrored block through a
// shared-memory transpose, so every global access is coalesced.
__global__ void __launch_bounds__(256)
isw_loss_grad_kernel(const float* __restrict__ f_cor, const float* __restrict__ mask, const float* __restrict__ off,
                     const float* __restrict__ num_remove, const float* __restrict__ grad_loss, int c, int hw,
                     int batch, float* __restrict__ s_out, float* __restrict__ alpha_out) {
    __shared__ float tr[32][33];
    const int b = blockIdx.z;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
    const float* fc = f_cor + (size_t)b * c * c;
    const float nr = num_remove[0];
    const float gate = (off[b] / nr >= 0.f) ? 1.f : 0.f;
    auto term = [&](int r, int q) {
        if (r >= c || q >= c) return 0.f;
        const float m = mask[(size_t)r * c + q];
        const float v = fc[(size_t)r * c + q] * m;
        const float sg = v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f);
        return sg * m;
    };
#pragma unroll
    for (int r = 0; r < 4; ++r) tr[ty + 8 * r][tx] = term(j0 + ty + 8 * r, i0 + tx);  // mirrored block, row-wise
    __syncthreads();
    const float scale = grad_loss[0] * gate / (nr * (float)batch) / (float)(hw - 1);
    if (alpha_out && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) alpha_out[b] = scale;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = i0 + ty + 8 * r, j = j0 + tx;
        if (i >= c || j >= c) continue;
        const float t = term(i, j) + tr[tx][ty + 8 * r];
        // alpha_out: factored form S_b = alpha_b * T_b for the tensor-core GEMM -- T is in {0, +-1, +-2} for a 0/1
        // mask, exact in TF32, which lets isw_sx_tc_kernel<EXACT> skip the hi/lo split of A
        s_out[(size_t)b * c * c + (size_t)i * c + j] = alpha_out ? t : scale * t;
    }
}

// S_b = (dF_b + dF_b^T) / (hw-1): backward of get_covariance_matrix for an arbitrary upstream gradient.
__global__ void __launch_bounds__(256)
isw_cov_grad_kernel(const float* __restrict__ d_fcor, int c, int hw, float* __restrict__ s_out) {
    const int b = blockIdx.y;
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= c * c) return;
    const int i = e / c, j = e % c;
    const float* d = d_fcor + (size_t)b * c * c;
    s_out[(size_t)b * c * c + e] = (d[(size_t)i * c + j] + d[(size_t)j * c + i]) / (float)(hw - 1);
}

// cal_covstat (models/ISW/__init__.py:93-104): var over the batch (unbiased, torch.var default) of the
// masked covariance f_cor * reverse_eye -- the statistic CovMatrix_ISW accumulates to pick its mask.
__global__ void __launch_bounds__(256)
isw_covstat_var_kernel(const float* __restrict__ f_cor, const float* __restrict__ reverse_eye, int batch, int cc,
                       float* __restrict__ var_out) {
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= cc) return;
    const float m = reverse_eye[e];
    float mean = 0.f;
    for (int b = 0; b < batch; ++b) mean += f_cor[(size_t)b * cc + e] * m;
    mean /= (float)batch;
    float ss = 0.f;
    for (int b = 0; b < batch; ++b) {
        const float d = f_cor[(size_t)b * cc + e] * m - mean;
        ss = fmaf(d, d, ss);
    }
    var_out[e] = ss / (float)(batch - 1);  // batch == 1 -> 0/0 = nan, like torch.var
}

// ------------------------------------------------------------- auxiliary Gram losses (SURVEY 8f rank 4)
// lw_loss (losses/lw.py:5-18): per-(n,c) standardisation with the UNBIASED variance and a true division by
// sqrt(var + 1e-5), optional spatial mask, Gram, sum of the squared strictly-upper-triangular entries.
// ortho_loss (losses/ortho.py:5-11): mean over C*C of triu(x y^T, 1)^2.  Both reuse the Gram / dX = S X kernels.

// One CTA per (n, c) plane.  yhat = standardised plane (kept for the backward), ym = yhat * mask (the Gram input;
// not written when there is no mask: ym == yhat).
// STATS (half-precision x, lw_loss's native route): only mean, sd and invstd of the plane are written -- the values the
// fp32 instantiation computes on the upcast plane; the fused Gram and dY = S Y standardise on load from them.
template <typename T, bool STATS>
__global__ void __launch_bounds__(NORM_THREADS)
lw_standardize_fwd_kernel(const T* __restrict__ x, const float* __restrict__ mask, int channels, int hw, float eps,
                          float* __restrict__ yhat, float* __restrict__ ym, float* __restrict__ invstd_out,
                          float* __restrict__ mean_out, float* __restrict__ sd_out) {
    __shared__ float scratch[NORM_THREADS / 32];
    const size_t base = (size_t)blockIdx.x * hw;
    float s = 0.f;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) s += Elem<T>::load(x[base + i]);
    const float mean = block_sum(s, scratch) / (float)hw;
    float q = 0.f;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float d = Elem<T>::load(x[base + i]) - mean;
        q = fmaf(d, d, q);
    }
    const float var = block_sum(q, scratch) / (float)(hw - 1);  // torch.var: unbiased; hw == 1 -> nan like torch
    const float sd = sqrtf(var + eps);
    if constexpr (STATS) {
        if (threadIdx.x == 0) {
            mean_out[blockIdx.x] = mean;
            sd_out[blockIdx.x] = sd;
            invstd_out[blockIdx.x] = 1.0f / sd;
        }
        return;
    }
    const float* mrow = mask ? mask + (size_t)(blockIdx.x / channels) * hw : nullptr;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float v = (Elem<T>::load(x[base + i]) - mean) / sd;
        yhat[base + i] = v;
        if (mrow) ym[base + i] = v * mrow[i];
    }
    if (threadIdx.x == 0) invstd_out[blockIdx.x] = 1.0f / sd;
}

// g = dy * mask; dx = (g - mean(g) - yhat * sum(g * yhat) / (hw - 1)) / sd
__global__ void __launch_bounds__(NORM_THREADS)
lw_standardize_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ yhat, const float* __restrict__ invstd,
                          const float* __restrict__ mask, int channels, int hw, float* __restrict__ dx) {
    __shared__ float scratch[NORM_THREADS / 32];
    const size_t base = (size_t)blockIdx.x * hw;
    const float* mrow = mask ? mask + (size_t)(blockIdx.x / channels) * hw : nullptr;
    float s1 = 0.f, s2 = 0.f;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float g = mrow ? dy[base + i] * mrow[i] : dy[base + i];
        s1 += g;
        s2 = fmaf(g, yhat[base + i], s2);
    }
    const float m1 = block_sum(s1, scratch) / (float)hw;
    const float m2 = block_sum(s2, scratch) / (float)(hw - 1);
    const float is = invstd[blockIdx.x];
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float g = mrow ? dy[base + i] * mrow[i] : dy[base + i];
        dx[base + i] = is * (g - m1 - yhat[base + i] * m2);
    }
}

// The same for a half-precision x: yhat is recomputed from x, mean and sd with the forward's operations ((x - mean) / sd:
// a sub and a true division, nothing to contract), so it is the fp32 route's yhat bit for bit; dx is written as RN(dx).
template <typename T>
__global__ void __launch_bounds__(NORM_THREADS)
lw_standardize_bwd_half_kernel(const float* __restrict__ dy, const T* __restrict__ x, const float* __restrict__ mean,
                               const float* __restrict__ sd, const float* __restrict__ invstd, const float* __restrict__ mask,
                               int channels, int hw, T* __restrict__ dx) {
    __shared__ float scratch[NORM_THREADS / 32];
    const size_t base = (size_t)blockIdx.x * hw;
    const float* mrow = mask ? mask + (size_t)(blockIdx.x / channels) * hw : nullptr;
    const float mu = mean[blockIdx.x], sdv = sd[blockIdx.x];
    // the rounding sequence is spelled out: it is the one nvcc compiles lw_standardize_bwd_kernel to (g = dy * m rounded
    // in the sums; g - m1 contracted to fma(dy, m, -m1) in the output, then fma(yhat, -m2, .) and the product with is)
    float s1 = 0.f, s2 = 0.f;
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float g = mrow ? __fmul_rn(dy[base + i], mrow[i]) : dy[base + i];
        s1 = __fadd_rn(s1, g);
        s2 = __fmaf_rn(g, __fdiv_rn(__fsub_rn(Elem<T>::load(x[base + i]), mu), sdv), s2);
    }
    const float m1 = block_sum(s1, scratch) / (float)hw;
    const float m2 = block_sum(s2, scratch) / (float)(hw - 1);
    const float is = invstd[blockIdx.x];
    for (int i = threadIdx.x; i < hw; i += NORM_THREADS) {
        const float t = mrow ? __fmaf_rn(dy[base + i], mrow[i], -m1) : __fsub_rn(dy[base + i], m1);
        const float yhat = __fdiv_rn(__fsub_rn(Elem<T>::load(x[base + i]), mu), sdv);
        dx[base + i] = Elem<T>::store(__fmul_rn(is, __fmaf_rn(yhat, -m2, t)));
    }
}

// Sum over the strictly-upper-triangular entries of g[rows 0..c) x cols col0..col0+c) (leading dimension ld) of
// every sample, squared; sliced like isw_loss_kernel, ordered final sum; loss = scale * total.
__global__ void __launch_bounds__(256)
triu_sq_loss_kernel(const float* __restrict__ g, int c, int ld, int col0, size_t sample_stride, int batch, float scale,
                    float* __restrict__ part, float* __restrict__ loss_out, unsigned int* __restrict__ ticket) {
    __shared__ float scratch[8];
    __shared__ bool s_last;
    const int b = blockIdx.y, chunks = gridDim.x;
    const float* gb = g + (size_t)b * sample_stride;
    const int rows_per = ceil_div(c, chunks);
    const int r0 = blockIdx.x * rows_per, r1 = min(c, r0 + rows_per);
    float s = 0.f;
    for (int i = r0; i < r1; ++i)
        for (int j = i + 1 + threadIdx.x; j < c; j += 256) {
            const float v = gb[(size_t)i * ld + col0 + j];
            s = fmaf(v, v, s);
        }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += scratch[w];
        part[b * LOSS_CHUNKS + blockIdx.x] = t;
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == (unsigned)(batch * chunks) - 1u;
    }
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    const volatile float* pv = part;
    float total = 0.f;
    for (int i = 0; i < batch; ++i)
        for (int k = 0; k < chunks; ++k) total += pv[i * LOSS_CHUNKS + k];
    loss_out[0] = scale * total;
    *ticket = 0u;
}

// lw backward: S_b = dG_b + dG_b^T with dG_b = 2 g triu(G_b, 1): symmetric, zero diagonal; the upper entry is used
// on both sides.
__global__ void __launch_bounds__(256)
lw_grad_s_kernel(const float* __restrict__ gram, const float* __restrict__ grad_loss, int c, float* __restrict__ s_out) {
    const int b = blockIdx.y;
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= c * c) return;
    const int i = e / c, j = e % c;
    const float* gb = gram + (size_t)b * c * c;
    const float v = i == j ? 0.f : gb[(size_t)min(i, j) * c + max(i, j)];
    s_out[(size_t)b * c * c + e] = 2.f * grad_loss[0] * v;
}

// ortho backward: Sx = (2 g / C^2) triu(G, 1) (dL/dx = Sx y) and Sy = Sx^T (dL/dy = Sy x); G is the block
// rows 0..c x cols c..2c of the stacked Gram (leading dimension 2c).
__global__ void __launch_bounds__(256)
ortho_grad_s_kernel(const float* __restrict__ gram_zz, const float* __restrict__ grad_loss, int c, float* __restrict__ sx,
                    float* __restrict__ sy) {
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= c * c) return;
    const int i = e / c, j = e % c;
    const float k = 2.f * grad_loss[0] / ((float)c * (float)c);
    sx[e] = j > i ? k * gram_zz[(size_t)i * 2 * c + c + j] : 0.f;
    sy[e] = i > j ? k * gram_zz[(size_t)j * 2 * c + c + i] : 0.f;
}

// ------------------------------------------------------------------------ top-k mask (CovMatrix_ISW)
// set_mask_matrix (models/ISW/cov_settings.py:52-72): mask = 1 at the k largest entries of the averaged
// variance matrix, 0 elsewhere, AND-ed with the previous mask.  The statistics are accumulated and averaged
// here too: values[i] = sum_s stats[s][i] / count, summed in arrival order like the reference's
// `var_matrix + var_cov` chain.  One CTA: MSB-first radix select of the k-th largest key (4 passes of 8 bits),
// then one ordered pass; ties at the threshold are taken in index order (torch.topk leaves tie order open).
constexpr int TOPK_THREADS = 1024;

__device__ __forceinline__ unsigned ordered_key(float v) {  // larger float <=> larger unsigned key
    const unsigned b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__global__ void __launch_bounds__(TOPK_THREADS)
isw_topk_mask_kernel(const float* __restrict__ stats, int n_stats, float count, int n, int k,
                     const float* __restrict__ prev_mask, float* __restrict__ values, float* __restrict__ mask) {
    __shared__ unsigned hist[256];
    __shared__ unsigned s_prefix;
    __shared__ int s_remaining;
    __shared__ int warp_cnt[TOPK_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < n; i += TOPK_THREADS) {
        float v = stats[i];
        for (int s = 1; s < n_stats; ++s) v = __fadd_rn(v, stats[(size_t)s * n + i]);
        values[i] = __fdiv_rn(v, count);
    }
    __syncthreads();
    unsigned prefix = 0, known = 0;
    int remaining = min(k, n);
    if (remaining > 0) {
        for (int shift = 24; shift >= 0; shift -= 8) {
            if (tid < 256) hist[tid] = 0;
            __syncthreads();
            for (int i = tid; i < n; i += TOPK_THREADS) {
                const unsigned key = ordered_key(values[i]);
                if ((key & known) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
            }
            __syncthreads();
            if (tid == 0) {
                int cum = 0, digit = 0;
                for (int b = 255; b >= 0; --b) {
                    if (cum + (int)hist[b] >= remaining) { digit = b; break; }
                    cum += (int)hist[b];
                }
                DGVCC_DEV_CHECK(remaining - cum >= 1 && remaining - cum <= (int)hist[digit]);   // the k-th key exists
                s_prefix = prefix | ((unsigned)digit << shift);
                s_remaining = remaining - cum;
            }
            __syncthreads();
            prefix = s_prefix;
            remaining = s_remaining;
            known |= 0xffu << shift;
        }
    }
    // prefix = key of the k-th largest; `remaining` of the entries equal to it are still to be taken
    int taken = 0;
    for (int base = 0; base < n; base += TOPK_THREADS) {
        const int i = base + tid;
        const unsigned key = i < n ? ordered_key(values[i]) : 0u;
        const bool gt = k > 0 && i < n && key > prefix, eq = k > 0 && i < n && key == prefix;
        const unsigned bal = __ballot_sync(FULL_MASK, eq);
        __syncthreads();
        if (lane == 0) warp_cnt[warp] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < TOPK_THREADS / 32; ++w) {
            if (w < warp) before += warp_cnt[w];
            total += warp_cnt[w];
        }
        const bool sel = gt || (eq && taken + before + __popc(bal & ((1u << lane) - 1u)) < remaining);
        if (i < n) mask[i] = (sel && (!prev_mask || prev_mask[i] != 0.f)) ? 1.f : 0.f;
        taken += total;
    }
}

// ------------------------------------------------------------------------------- dX = S X (SIMT)
__global__ void __launch_bounds__(GEMM_THREADS)
isw_sx_simt_kernel(const float* __restrict__ s, const float* __restrict__ x, int c, int hw, float* __restrict__ dx) {
    __shared__ float as[GK][GT + 4];  // S tile, transposed: as[k][row]
    __shared__ float bs[GK][GT + 4];  // X tile: bs[k][col]
    const int b = blockIdx.z;
    const int row0 = blockIdx.y * GT, col0 = blockIdx.x * GT;
    const float* sb = s + (size_t)b * c * c;
    const float* xb = x + (size_t)b * c * hw;
    const int tid = threadIdx.x;
    const int lr = tid >> 2, lk = (tid & 3) * 4;   // S loader
    const int xk = tid >> 4, xc = (tid & 15) * 4;  // X loader: row xk of the chunk, 4 consecutive columns
    const int ty = tid >> 4, tx = tid & 15;
    float acc[4][4] = {};
    for (int kb = 0; kb < c; kb += GK) {
        float pa[4], pb[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int r = row0 + lr, k = kb + lk + q;
            pa[q] = (r < c && k < c) ? sb[(size_t)r * c + k] : 0.f;
            const int kk = kb + xk, col = col0 + xc + q;
            pb[q] = (kk < c && col < hw) ? xb[(size_t)kk * hw + col] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) { as[lk + q][lr] = pa[q]; bs[xk][xc + q] = pb[q]; }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < GK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&as[k][ty * 4]);
            const float4 bb = *reinterpret_cast<const float4*>(&bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
    }
    float* out = dx + (size_t)b * c * hw;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = row0 + ty * 4 + i;
        if (r >= c) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int col = col0 + tx * 4 + j;
            if (col < hw) out[(size_t)r * hw + col] = acc[i][j];
        }
    }
}

}  // namespace isw
}  // namespace dgvcc

using namespace dgvcc;
using namespace dgvcc::isw;

// Dynamic shared memory a launch of isw_instnorm_fwd_kernel gets without the opt-in.  The kernel's static shared memory
// (its scratch, plus the 1 KB the runtime reserves per block: 1056 bytes in `cuobjdump -res-usage`) counts against the
// same 48 KB, so a 48 KB plane needs the opt-in too; 2 KB of slack keeps the rule clear of the static size.
constexpr size_t NORM_SMEM_NO_OPT_IN = 48 * 1024 - 2048;

template <typename T>
static int instnorm_forward(const T* x, int planes, int hw, float eps, T* y, float* mean, float* invstd, void* stream) {
    const size_t smem = (size_t)hw * sizeof(T);
    const bool fits = smem <= 200 * 1024;
    if (fits && smem > NORM_SMEM_NO_OPT_IN) {  // opt in once per device to the largest plane the kernel caches (not per call: the
                                     // call is not allowed while a stream is being captured into a CUDA graph)
        static PerDeviceOnce once;
        if (once.first())
            DGVCC_RETURN_IF_CUDA(cudaFuncSetAttribute(isw_instnorm_fwd_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                      200 * 1024));
    }
    // gridDim.y == 2 tells the kernel the plane is not cached (only y-block 0 writes)
    isw_instnorm_fwd_kernel<T><<<dim3(planes, fits ? 1 : 2), NORM_THREADS, fits ? smem : 0, (cudaStream_t)stream>>>(
        x, hw, eps, y, mean, invstd);
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_isw_instnorm_forward(const float* x, int planes, int hw, float eps, float* y, float* mean,
                                          float* invstd, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !y || !mean || !invstd || planes <= 0 || hw <= 0) return DGVCC_ERR_ARG;
    return instnorm_forward(x, planes, hw, eps, y, mean, invstd, stream);
}

// The fp16 / bf16 dispatch of the *_h entry points: runs the statements `...` with T the element type dtype names, and
// returns DGVCC_ERR_ARG for any other dtype.  A macro rather than a function template over a generic lambda, so a kernel
// template launched in the statements is instantiated where it stands and the kernels keep their order in the object.
#define DGVCC_BY_HALF_DTYPE(dtype, ...)                                                          \
    do {                                                                                         \
        if ((dtype) == DGVCC_DTYPE_F16) { using T = __half; __VA_ARGS__ }                        \
        else if ((dtype) == DGVCC_DTYPE_BF16) { using T = __nv_bfloat16; __VA_ARGS__ }           \
        else return DGVCC_ERR_ARG;                                                               \
    } while (0)

extern "C" int dgvcc_isw_instnorm_forward_h(const void* x, int dtype, int planes, int hw, float eps, void* y, float* mean,
                                            float* invstd, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !y || !mean || !invstd || planes <= 0 || hw <= 0) return DGVCC_ERR_ARG;
    DGVCC_BY_HALF_DTYPE(dtype, return instnorm_forward((const T*)x, planes, hw, eps, (T*)y, mean, invstd, stream););
}

extern "C" int dgvcc_isw_instnorm_backward_h(const void* dy, const void* x, const float* mean, const float* invstd, int dtype,
                                             int planes, int hw, void* dx, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!dy || !x || !mean || !invstd || !dx || planes <= 0 || hw <= 0) return DGVCC_ERR_ARG;
    DGVCC_BY_HALF_DTYPE(dtype, isw_instnorm_bwd_half_kernel<<<planes, NORM_THREADS, 0, (cudaStream_t)stream>>>(
                                   (const T*)dy, (const T*)x, mean, invstd, hw, (T*)dx););
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_isw_instnorm_backward(const float* dy, const float* y, const float* invstd, int planes, int hw,
                                           float* dx, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!dy || !y || !invstd || !dx || planes <= 0 || hw <= 0) return DGVCC_ERR_ARG;
    isw_instnorm_bwd_kernel<<<planes, NORM_THREADS, 0, (cudaStream_t)stream>>>(dy, y, invstd, hw, dx);
    return (int)cudaGetLastError();
}

// Split-K plans.  SIMT Gram: 64x64 tiles, enough CTAs to cover the chip about twice.  Tensor-core Gram: one CTA
// per SM and one wave (the kernel bounds its in-TMEM accumulation chains itself, so K per CTA may be long);
// C <= 64 packs two samples into one 128-row tile and stores 64x64 partial tiles.
// Shapes the ISW-family launchers accept (the reference's are (8, 64..512, 1600..25 600)); beyond them the int
// arithmetic of the plans and grids would overflow.  batch is a grid z dimension (<= 65535).
static bool isw_shape_ok(int batch, int c, int hw) {
    return batch >= 1 && batch <= 65535 && c >= 1 && c <= 32768 && hw >= 1 && hw <= (1 << 30);
}

static void gram_plan_simt(int batch, int c, int hw, int* splits, int* k_per_split, int* n_tiles) {
    const int t1 = ceil_div(c, 64);
    *n_tiles = t1 * (t1 + 1) / 2;
    const long long work = (long long)batch * *n_tiles;
    int s = work >= 296 ? 1 : ceil_div(296, (int)work);
    const int max_s = ceil_div(hw, 256);
    if (s > max_s) s = max_s;
    if (s < 1) s = 1;
    const int kps = ceil_div(ceil_div(hw, s), 32) * 32;
    *splits = ceil_div(hw, kps);
    *k_per_split = kps;
}

static void gram_plan_tc(int batch, int c, int hw, int* splits, int* k_per_split, int* n_tiles, int* tile) {
    const bool pair = c <= 64;
    *tile = pair ? 64 : 128;
    const int t1 = pair ? 1 : ceil_div(c, 128);
    *n_tiles = t1 * (t1 + 1) / 2;
    const long long units = (long long)(pair ? ceil_div(batch, 2) : batch) * *n_tiles;
    int s = units > 148 ? 0 : (int)(148 / units);
    const int max_s = ceil_div(hw, 256);
    if (s > max_s) s = max_s;
    if (s < 1) s = 1;
    const int kps = ceil_div(ceil_div(hw, s), 32) * 32;
    *splits = ceil_div(hw, kps);
    *k_per_split = kps;
}

static size_t gram_partial_floats(int batch, int c, int hw) {
    int s, k, n, tile;
    gram_plan_simt(batch, c, hw, &s, &k, &n);
    const size_t p_simt = (size_t)batch * s * n * 64 * 64;
    gram_plan_tc(batch, c, hw, &s, &k, &n, &tile);
    const size_t p_tc = (size_t)batch * s * n * tile * tile;
    return p_simt > p_tc ? p_simt : p_tc;
}

extern "C" size_t dgvcc_isw_workspace_bytes(int batch, int c, int hw) {
    if (!isw_shape_ok(batch, c, hw)) return 0;   // the launchers reject such shapes (the split plans divide by them)
    // partials | off[B] + loss partials [B][LOSS_CHUNKS] + alpha[B] | ticket (256 B) | S [B,C,C]
    return align_up(gram_partial_floats(batch, c, hw) * sizeof(float), 256) +
           align_up((size_t)batch * (2 + LOSS_CHUNKS) * sizeof(float), 256) +
           256 + align_up((size_t)batch * c * c * sizeof(float), 256);
}

namespace {
struct IswWs { float* part; float* off; float* alpha; unsigned int* ticket; float* s; };
IswWs carve(void* ws, int batch, int c, int hw) {
    const size_t part = align_up(gram_partial_floats(batch, c, hw) * sizeof(float), 256);
    IswWs w;
    char* p = (char*)ws;
    w.part = (float*)p; p += part;
    w.off = (float*)p; p += align_up((size_t)batch * (2 + LOSS_CHUNKS) * sizeof(float), 256);
    w.alpha = w.off + (size_t)batch * (1 + LOSS_CHUNKS);
    w.ticket = (unsigned int*)p; p += 256;
    w.s = (float*)p;
    return w;
}
}  // namespace

template <typename T> constexpr bool HALF = !std::is_same<T, float>::value;

// Gram of every sample, finished as out = X X^T / denom (+ eps * eye when eye is given).  The tensor-core partials where
// the shape tiles; else exact fp32 on CUDA cores for an fp32 map, and DGVCC_ERR_UNSUPPORTED for a half one.  STD: the Gram
// of lw's standardised map (x - mean) / sd (* mask), computed from the half x.
template <typename T, bool STD = false>
static int launch_gram(const T* x, const float* mean, const float* sd, const float* mask, const float* eye, float denom,
                       float eps, int batch, int c, int hw, int use_tensor_cores, const IswWs& w, float* out, cudaStream_t st) {
    int splits, kps, n_tiles, tile = 64;
    int rc = DGVCC_ERR_UNSUPPORTED;
    if (use_tensor_cores) {
        gram_plan_tc(batch, c, hw, &splits, &kps, &n_tiles, &tile);
        rc = isw_tc::launch<T, STD>(x, mean, sd, mask, batch, c, hw, splits, kps, w.part, st);
    }
    if constexpr (!HALF<T>) {
        if (rc == DGVCC_ERR_UNSUPPORTED) {
            tile = 64;
            gram_plan_simt(batch, c, hw, &splits, &kps, &n_tiles);
            isw_gram_simt_kernel<<<dim3(n_tiles, splits, batch), GEMM_THREADS, 0, st>>>(x, c, hw, splits, kps, w.part);
            rc = (int)cudaGetLastError();
        }
    }
    if (rc != DGVCC_OK) return rc;
    const int yblocks = (tile / 32) * (tile / 32);
    isw_cov_finish_kernel<<<dim3(n_tiles, yblocks, batch), 256, 0, st>>>(w.part, c, denom, splits, tile, eye, eps, out);
    return (int)cudaGetLastError();
}

// dX = S X on the tensor cores where the shape tiles; else exact fp32 on CUDA cores for an fp32 X, and
// DGVCC_ERR_UNSUPPORTED for a half one.
template <typename T>
static int launch_sx(const float* s, const void* x, int batch, int c, int hw, int use_tensor_cores, void* dx, cudaStream_t st) {
    int rc = DGVCC_ERR_UNSUPPORTED;
    if (use_tensor_cores)
        rc = isw_sx::launch<T>(s, (const T*)x, nullptr, nullptr, nullptr, batch, c, hw, dx, nullptr, false, st);
    if constexpr (!HALF<T>) {
        if (rc == DGVCC_ERR_UNSUPPORTED) {
            isw_sx_simt_kernel<<<dim3(ceil_div(hw, GT), ceil_div(c, GT), batch), GEMM_THREADS, 0, st>>>(s, (const float*)x, c,
                                                                                                      hw, (float*)dx);
            rc = (int)cudaGetLastError();
        }
    }
    return rc;
}

// A half dX = S X has no CUDA-core fallback, so the half backwards refuse a shape the tensor cores do not tile before they
// compute S (the launcher checks the rule again, S's base included).
template <typename T> static bool half_untiled(const void* x, const void* dx, int c, int hw) {
    return HALF<T> && !(half_tc_tiles(c, hw) && tma_aligned(x, dx));
}

// The fp32 and half (*_h) entry points share one body per pair, templated over the element type T of the map and its
// gradient.  The half types run on the tensor cores only (use_tensor_cores = 1) and return DGVCC_ERR_UNSUPPORTED where
// fp32 falls back to the CUDA cores; every value is the one the fp32 path computes on the upcast map (DESIGN section 5).
template <typename T>
static int covariance(const void* f_map, const float* eye, int batch, int c, int hw, int use_tensor_cores, void* workspace,
                      size_t workspace_bytes, float* f_cor, void* stream) {
    if (!f_map || !eye || !workspace || !f_cor || !isw_shape_ok(batch, c, hw) || hw <= 1) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_isw_workspace_bytes(batch, c, hw)) return DGVCC_ERR_WORKSPACE;
    return launch_gram((const T*)f_map, nullptr, nullptr, nullptr, eye, (float)(hw - 1), 1e-5f, batch, c, hw, use_tensor_cores,
                       carve(workspace, batch, c, hw), f_cor, (cudaStream_t)stream);
}

extern "C" int dgvcc_isw_covariance(const float* f_map, const float* eye, int batch, int c, int hw, int use_tensor_cores,
                                    void* workspace, size_t workspace_bytes, float* f_cor, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    return covariance<float>(f_map, eye, batch, c, hw, use_tensor_cores, workspace, workspace_bytes, f_cor, stream);
}

extern "C" int dgvcc_isw_covariance_h(const void* f_map, int dtype, const float* eye, int batch, int c, int hw,
                                      void* workspace, size_t workspace_bytes, float* f_cor, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    DGVCC_BY_HALF_DTYPE(dtype, return covariance<T>(f_map, eye, batch, c, hw, 1, workspace, workspace_bytes, f_cor, stream););
}

extern "C" int dgvcc_isw_loss_forward(const float* f_cor, const float* mask, const float* margin,
                                      const float* num_remove_cov, int batch, int c, int hw, void* workspace,
                                      size_t workspace_bytes, float* loss_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!f_cor || !mask || !margin || !num_remove_cov || !workspace || !loss_out || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_isw_workspace_bytes(batch, c, hw)) return DGVCC_ERR_WORKSPACE;
    const IswWs w = carve(workspace, batch, c, hw);
    cudaStream_t st = (cudaStream_t)stream;
    DGVCC_RETURN_IF_CUDA(cudaMemsetAsync(w.ticket, 0, sizeof(unsigned int), st));
    const int chunks = max(1, min(LOSS_CHUNKS, c * c / 4096));
    isw_loss_kernel<<<dim3(chunks, batch), 256, 0, st>>>(f_cor, mask, c, batch, margin, num_remove_cov, w.off, loss_out,
                                                        w.ticket);
    return (int)cudaGetLastError();
}

template <typename T>
static int loss_backward(const void* f_map, const float* f_cor, const float* mask, const float* num_remove_cov,
                         const float* grad_loss, int batch, int c, int hw, int use_tensor_cores, int mask_is_binary,
                         void* workspace, size_t workspace_bytes, void* grad_f_map, void* stream) {
    if (!f_map || !f_cor || !mask || !num_remove_cov || !grad_loss || !workspace || !grad_f_map || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_isw_workspace_bytes(batch, c, hw)) return DGVCC_ERR_WORKSPACE;
    if (half_untiled<T>(f_map, grad_f_map, c, hw)) return DGVCC_ERR_UNSUPPORTED;
    const IswWs w = carve(workspace, batch, c, hw);
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 s_grid(ceil_div(c, 32), ceil_div(c, 32), batch);
    if (mask_is_binary && (HALF<T> || (use_tensor_cores && sx_tc_tiles(c, hw) && tma_aligned(w.s, f_map, grad_f_map)))) {
        // factored S = alpha * T: the GEMM runs on T (TF32-exact for a 0/1 mask) and scales in its epilogue
        isw_loss_grad_kernel<<<s_grid, 256, 0, st>>>(f_cor, mask, w.off, num_remove_cov, grad_loss, c, hw, batch, w.s, w.alpha);
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
        const int rc = isw_sx::launch<T>(w.s, (const T*)f_map, nullptr, nullptr, nullptr, batch, c, hw, grad_f_map, w.alpha,
                                         true, st);
        if (HALF<T> || rc != DGVCC_ERR_UNSUPPORTED) return rc;
    }
    isw_loss_grad_kernel<<<s_grid, 256, 0, st>>>(f_cor, mask, w.off, num_remove_cov, grad_loss, c, hw, batch, w.s, nullptr);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return launch_sx<T>(w.s, f_map, batch, c, hw, use_tensor_cores, grad_f_map, st);
}

extern "C" int dgvcc_isw_loss_backward(const float* f_map, const float* f_cor, const float* mask,
                                       const float* num_remove_cov, const float* grad_loss, int batch, int c, int hw,
                                       int use_tensor_cores, int mask_is_binary, void* workspace,
                                       size_t workspace_bytes, float* grad_f_map, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    return loss_backward<float>(f_map, f_cor, mask, num_remove_cov, grad_loss, batch, c, hw, use_tensor_cores, mask_is_binary,
                                workspace, workspace_bytes, grad_f_map, stream);
}

extern "C" int dgvcc_isw_loss_backward_h(const void* f_map, int dtype, const float* f_cor, const float* mask,
                                         const float* num_remove_cov, const float* grad_loss, int batch, int c, int hw,
                                         int mask_is_binary, void* workspace, size_t workspace_bytes, void* grad_f_map,
                                         void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    DGVCC_BY_HALF_DTYPE(dtype, return loss_backward<T>(f_map, f_cor, mask, num_remove_cov, grad_loss, batch, c, hw, 1,
                                                       mask_is_binary, workspace, workspace_bytes, grad_f_map, stream););
}

template <typename T>
static int covariance_backward(const void* f_map, const float* grad_f_cor, int batch, int c, int hw, int use_tensor_cores,
                               void* workspace, size_t workspace_bytes, void* grad_f_map, void* stream) {
    if (!f_map || !grad_f_cor || !workspace || !grad_f_map || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_isw_workspace_bytes(batch, c, hw)) return DGVCC_ERR_WORKSPACE;
    if (half_untiled<T>(f_map, grad_f_map, c, hw)) return DGVCC_ERR_UNSUPPORTED;
    const IswWs w = carve(workspace, batch, c, hw);
    cudaStream_t st = (cudaStream_t)stream;
    isw_cov_grad_kernel<<<dim3(ceil_div(c * c, 256), batch), 256, 0, st>>>(grad_f_cor, c, hw, w.s);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return launch_sx<T>(w.s, f_map, batch, c, hw, use_tensor_cores, grad_f_map, st);
}

extern "C" int dgvcc_isw_covariance_backward(const float* f_map, const float* grad_f_cor, int batch, int c, int hw,
                                             int use_tensor_cores, void* workspace, size_t workspace_bytes,
                                             float* grad_f_map, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    return covariance_backward<float>(f_map, grad_f_cor, batch, c, hw, use_tensor_cores, workspace, workspace_bytes,
                                      grad_f_map, stream);
}

extern "C" int dgvcc_isw_covariance_backward_h(const void* f_map, int dtype, const float* grad_f_cor, int batch, int c,
                                               int hw, void* workspace, size_t workspace_bytes, void* grad_f_map,
                                               void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    DGVCC_BY_HALF_DTYPE(dtype, return covariance_backward<T>(f_map, grad_f_cor, batch, c, hw, 1, workspace, workspace_bytes,
                                                             grad_f_map, stream););
}

extern "C" int dgvcc_isw_covstat_var(const float* f_cor, const float* reverse_eye, int batch, int c, float* var_out,
                                     void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!f_cor || !reverse_eye || !var_out || batch <= 0 || c <= 0) return DGVCC_ERR_ARG;
    isw_covstat_var_kernel<<<ceil_div(c * c, 256), 256, 0, (cudaStream_t)stream>>>(f_cor, reverse_eye, batch, c * c, var_out);
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_isw_topk_mask(const float* stats, int n_stats, int count, int n, int k, const float* prev_mask,
                                   float* values, float* mask, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!stats || !values || !mask || n_stats <= 0 || count <= 0 || n <= 0 || k < 0) return DGVCC_ERR_ARG;
    isw_topk_mask_kernel<<<1, TOPK_THREADS, 0, (cudaStream_t)stream>>>(stats, n_stats, (float)count, n, k, prev_mask,
                                                                       values, mask);
    return (int)cudaGetLastError();
}

// ------------------------------------------------------------------ auxiliary Gram losses: entry points
extern "C" int dgvcc_lw_standardize_forward(const float* x, const float* mask, int batch, int c, int hw, float eps,
                                            float* yhat, float* y_masked, float* invstd, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !yhat || !invstd || batch <= 0 || c <= 0 || hw <= 0 || (mask && !y_masked)) return DGVCC_ERR_ARG;
    lw_standardize_fwd_kernel<float, false><<<batch * c, NORM_THREADS, 0, (cudaStream_t)stream>>>(x, mask, c, hw, eps, yhat,
                                                                                                  y_masked, invstd, nullptr,
                                                                                                  nullptr);
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_lw_standardize_backward(const float* dy, const float* yhat, const float* invstd, const float* mask,
                                             int batch, int c, int hw, float* dx, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!dy || !yhat || !invstd || !dx || batch <= 0 || c <= 0 || hw <= 0) return DGVCC_ERR_ARG;
    lw_standardize_bwd_kernel<<<batch * c, NORM_THREADS, 0, (cudaStream_t)stream>>>(dy, yhat, invstd, mask, c, hw, dx);
    return (int)cudaGetLastError();
}

template <typename T>
static int gram(const void* f_map, int batch, int c, int hw, int use_tensor_cores, void* workspace, size_t workspace_bytes,
                float* gram, void* stream) {
    if (!f_map || !workspace || !gram || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_isw_workspace_bytes(batch, c, hw)) return DGVCC_ERR_WORKSPACE;
    return launch_gram((const T*)f_map, nullptr, nullptr, nullptr, nullptr, 1.0f, 0.f, batch, c, hw, use_tensor_cores,
                       carve(workspace, batch, c, hw), gram, (cudaStream_t)stream);
}

extern "C" int dgvcc_isw_gram(const float* f_map, int batch, int c, int hw, int use_tensor_cores, void* workspace,
                              size_t workspace_bytes, float* gram, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    return ::gram<float>(f_map, batch, c, hw, use_tensor_cores, workspace, workspace_bytes, gram, stream);
}

extern "C" int dgvcc_isw_gram_h(const void* f_map, int dtype, int batch, int c, int hw, void* workspace,
                                size_t workspace_bytes, float* gram, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    DGVCC_BY_HALF_DTYPE(dtype, return ::gram<T>(f_map, batch, c, hw, 1, workspace, workspace_bytes, gram, stream););
}

static int launch_triu_sq(const float* g, int c, int ld, int col0, size_t sample_stride, int batch, float scale,
                          const IswWs& w, float* loss_out, cudaStream_t st) {
    DGVCC_RETURN_IF_CUDA(cudaMemsetAsync(w.ticket, 0, sizeof(unsigned int), st));
    const int chunks = max(1, min(LOSS_CHUNKS, c / 16));
    triu_sq_loss_kernel<<<dim3(chunks, batch), 256, 0, st>>>(g, c, ld, col0, sample_stride, batch, scale, w.off + batch,
                                                             loss_out, w.ticket);
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_lw_loss_forward(const float* gram, int batch, int c, int hw, void* workspace, size_t workspace_bytes,
                                     float* loss_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!gram || !workspace || !loss_out || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_isw_workspace_bytes(batch, c, hw)) return DGVCC_ERR_WORKSPACE;
    const IswWs w = carve(workspace, batch, c, hw);
    return launch_triu_sq(gram, c, c, 0, (size_t)c * c, batch, 1.0f, w, loss_out, (cudaStream_t)stream);
}

extern "C" int dgvcc_lw_loss_backward(const float* y, const float* gram, const float* grad_loss, int batch, int c, int hw,
                                      int use_tensor_cores, void* workspace, size_t workspace_bytes, float* grad_y,
                                      void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!y || !gram || !grad_loss || !workspace || !grad_y || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_isw_workspace_bytes(batch, c, hw)) return DGVCC_ERR_WORKSPACE;
    const IswWs w = carve(workspace, batch, c, hw);
    cudaStream_t st = (cudaStream_t)stream;
    lw_grad_s_kernel<<<dim3(ceil_div(c * c, 256), batch), 256, 0, st>>>(gram, grad_loss, c, w.s);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return launch_sx<float>(w.s, y, batch, c, hw, use_tensor_cores, grad_y, st);
}

// z = [x; y] stacked [2c, p]; gram_zz [2c, 2c] = z z^T from dgvcc_isw_gram(z, 1, 2c, p, ...).
extern "C" int dgvcc_ortho_loss_forward(const float* gram_zz, int c, int p, void* workspace, size_t workspace_bytes,
                                        float* loss_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!gram_zz || !workspace || !loss_out || c > 16384 || !isw_shape_ok(1, 2 * c, p)) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_isw_workspace_bytes(1, 2 * c, p)) return DGVCC_ERR_WORKSPACE;
    const IswWs w = carve(workspace, 1, 2 * c, p);
    return launch_triu_sq(gram_zz, c, 2 * c, c, 0, 1, 1.0f / ((float)c * (float)c), w, loss_out, (cudaStream_t)stream);
}

// x, y, grad_x, grad_y [c, p] of type T; gram_zz from the Gram of z = [x; y].
template <typename T>
static int ortho_loss_backward(const void* x, const void* y, const float* gram_zz, const float* grad_loss, int c, int p,
                               int use_tensor_cores, void* workspace, size_t workspace_bytes, void* grad_x, void* grad_y,
                               void* stream) {
    if (!x || !y || !gram_zz || !grad_loss || !workspace || !grad_x || !grad_y || c > 16384 || !isw_shape_ok(1, 2 * c, p)) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_isw_workspace_bytes(1, 2 * c, p)) return DGVCC_ERR_WORKSPACE;
    if (half_untiled<T>(x, grad_x, c, p) || half_untiled<T>(y, grad_y, c, p)) return DGVCC_ERR_UNSUPPORTED;
    const IswWs w = carve(workspace, 1, 2 * c, p);  // S region holds (2c)^2 floats: Sx and Sy fit
    cudaStream_t st = (cudaStream_t)stream;
    float* sx = w.s;
    float* sy = w.s + (size_t)c * c;
    ortho_grad_s_kernel<<<ceil_div(c * c, 256), 256, 0, st>>>(gram_zz, grad_loss, c, sx, sy);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    const int rc = launch_sx<T>(sx, y, 1, c, p, use_tensor_cores, grad_x, st);
    if (rc != DGVCC_OK) return rc;
    return launch_sx<T>(sy, x, 1, c, p, use_tensor_cores, grad_y, st);
}

extern "C" int dgvcc_ortho_loss_backward(const float* x, const float* y, const float* gram_zz, const float* grad_loss, int c,
                                         int p, int use_tensor_cores, void* workspace, size_t workspace_bytes,
                                         float* grad_x, float* grad_y, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    return ortho_loss_backward<float>(x, y, gram_zz, grad_loss, c, p, use_tensor_cores, workspace, workspace_bytes, grad_x,
                                      grad_y, stream);
}

extern "C" int dgvcc_ortho_loss_backward_h(const void* x, const void* y, int dtype, const float* gram_zz,
                                           const float* grad_loss, int c, int p, void* workspace, size_t workspace_bytes,
                                           void* grad_x, void* grad_y, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    DGVCC_BY_HALF_DTYPE(dtype, return ortho_loss_backward<T>(x, y, gram_zz, grad_loss, c, p, 1, workspace, workspace_bytes,
                                                             grad_x, grad_y, stream););
}

// ------------------------------------------------------- auxiliary Gram losses: half-precision entry points
// lw_loss on a half map, the standardised map never materialised: the values of the fp32 entry points above on the map
// upcast to fp32 (DESIGN section 5b); the Gram and dY = S Y run on the tensor cores only, under half_tc_tiles.

extern "C" int dgvcc_lw_standardize_stats_h(const void* x, int dtype, int batch, int c, int hw, float eps, float* mean,
                                            float* sd, float* invstd, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !mean || !sd || !invstd || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    DGVCC_BY_HALF_DTYPE(dtype, lw_standardize_fwd_kernel<T, true><<<batch * c, NORM_THREADS, 0, (cudaStream_t)stream>>>(
                                   (const T*)x, nullptr, c, hw, eps, nullptr, nullptr, invstd, mean, sd););
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_lw_gram_h(const void* x, int dtype, const float* mean, const float* sd, const float* mask, int batch,
                               int c, int hw, void* workspace, size_t workspace_bytes, float* gram, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !mean || !sd || !workspace || !gram || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    DGVCC_BY_HALF_DTYPE(dtype, {
        if (workspace_bytes < dgvcc_isw_workspace_bytes(batch, c, hw)) return DGVCC_ERR_WORKSPACE;
        return launch_gram<T, true>((const T*)x, mean, sd, mask, nullptr, 1.0f, 0.f, batch, c, hw, 1,
                                    carve(workspace, batch, c, hw), gram, (cudaStream_t)stream);
    });
}

extern "C" int dgvcc_lw_loss_backward_h(const void* x, int dtype, const float* mean, const float* sd, const float* mask,
                                        const float* gram, const float* grad_loss, int batch, int c, int hw, void* workspace,
                                        size_t workspace_bytes, float* grad_y, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !mean || !sd || !gram || !grad_loss || !workspace || !grad_y || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    DGVCC_BY_HALF_DTYPE(dtype, {
        if (workspace_bytes < dgvcc_isw_workspace_bytes(batch, c, hw)) return DGVCC_ERR_WORKSPACE;
        if (half_untiled<T>(x, grad_y, c, hw)) return DGVCC_ERR_UNSUPPORTED;
        const IswWs w = carve(workspace, batch, c, hw);
        cudaStream_t st = (cudaStream_t)stream;
        lw_grad_s_kernel<<<dim3(ceil_div(c * c, 256), batch), 256, 0, st>>>(gram, grad_loss, c, w.s);
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
        return isw_sx::launch<T, true>(w.s, (const T*)x, mean, sd, mask, batch, c, hw, grad_y, nullptr, false, st);
    });
}

extern "C" int dgvcc_lw_standardize_backward_h(const float* dy, const void* x, int dtype, const float* mean, const float* sd,
                                               const float* invstd, const float* mask, int batch, int c, int hw, void* dx,
                                               void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!dy || !x || !mean || !sd || !invstd || !dx || !isw_shape_ok(batch, c, hw)) return DGVCC_ERR_ARG;
    DGVCC_BY_HALF_DTYPE(dtype, lw_standardize_bwd_half_kernel<<<batch * c, NORM_THREADS, 0, (cudaStream_t)stream>>>(
                                   dy, (const T*)x, mean, sd, invstd, mask, c, hw, (T*)dx););
    return (int)cudaGetLastError();
}
