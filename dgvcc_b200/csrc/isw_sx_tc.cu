// ISW backward GEMM  dX_b = S_b X_b  on the Blackwell tensor cores (tcgen05 + TMEM + TMA).
//
// Autograd of models/ISW/instance_whitening.py:37: S_b [C,C] is the symmetrised upstream gradient of the
// covariance (already divided by HW-1), X_b [C,HW] the whitened map.  M = C rows of dX, N = HW columns,
// K = C.  A = S is K-major (k contiguous); B = X is MN-major (n contiguous).  The tensor core accepts
// MN-major TF32 operands only in the SWIZZLE_128B_BASE32B layout (atoms of 4 k-rows x 128 bytes whose
// 32-byte chunks are XOR-ed with the row index), which TMA produces with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
// X is staged as four 32(n) x 32(k) boxes per k block: 32-float n segments LBO = 4 KB apart, 4-row k
// groups SBO = 512 B apart.
// fp32 accuracy as in the Gram: 3xTF32, A and B both split into hi + lo, cross terms in their own TMEM
// accumulator.  The accumulation chain is only C/8 steps, so no split-K is needed.
// One CTA = one 128 x 128 tile of dX of one sample; warp roles as in isw_gram_tc.cu.
//
// EXACT variant (the backward of instance_whitening_loss): there S_b = alpha_b * T_b with T_b = sgn(.)*mask
// in {0, +-1, +-2} for a 0/1 mask -- exactly representable in TF32.  The caller passes T and alpha; A then
// needs neither conversion nor a lo part (2 MMAs per k step instead of 3, a third less shared-memory traffic),
// the stage shrinks to 48 KB so two CTAs share an SM (one's epilogue under the other's main loop), and the
// epilogue multiplies by alpha_b.  The caller promises exactness (`a_is_tf32_exact`: the Python side checks the
// mask once per mask tensor and caches the answer).
//
// Half-precision X (isw_sx_tc_kernel<EXACT, __half / __nv_bfloat16>): TMA loads X as one 32(k) x 128(n) half box (256-byte
// rows, no swizzle) at the end of the stage; the converters widen it into the SWIZZLE_128B_BASE32B fp32 B tile above
// (box j = n / 32 at j * 4 KB, k row kk at kk * 128 B, 32-byte chunk c at chunk c ^ (kk % 4)).  X_lo is exactly 0, so
// the MMAs on it go away: EXACT runs 1 MMA per k step (S X_hi), the general variant 2 (S_hi X_hi, and S_lo X_hi opening
// the cross accumulator).  dX is written rounded to nearest in the input's type.
//
// Standardise on load (isw_sx_tc_kernel<false, half, STD = true>, dY = S Y of lw_loss's backward): TMA loads the half X
// tile as above, and the converters compute  y = (x - mean_k) / sd_k  (times mask[n] under a mask) with the IEEE
// operations of lw_standardize_fwd_kernel, k being the channel, and write hi and lo = RN_tf32(y - trunc_tf32(y)) into the
// B_hi / B_lo tiles of the fp32 layout.  The MMAs and the fp32 epilogue are those of the fp32 general kernel, so dY is the
// same bits as dgvcc_isw_sx_tc on the materialised standardised map.  Channels k >= C and columns n >= hw are written as
// 0, what TMA zero-fills there for the fp32 kernel, without reading statistics or mask.
#include <type_traits>

#include "isw_tc.cuh"
#include "tc_common.cuh"
#include "../../include/dgvcc_b200.h"

namespace dgvcc {
namespace isw_sx {

using namespace dgvcc::tc;

constexpr int TILE = 128;                  // M and N of the output tile
constexpr int BLOCK_K = 32;
constexpr int UMMA_K = 8;
constexpr int TILE_BYTES = TILE * BLOCK_K * 4;  // 16 KB for either operand
constexpr int THREADS = 192;
constexpr int CONVERTER_WARPS = 4;
constexpr int HTILE_BYTES = TILE * BLOCK_K * 2;  // 8 KB: a half-precision X tile as TMA delivers it
template <bool EXACT, typename T = float, bool STD = false> struct Cfg {
    static constexpr bool HALF = !std::is_same<T, float>::value;
    static constexpr int STAGES = EXACT ? 2 : 3;
    // fp32: EXACT: A, B_hi, B_lo; else A_hi, B_hi, A_lo, B_lo.  half: the same without B_lo, then the half X tile (B_H).
    // STD (general only): A_hi, B_hi, A_lo, B_lo, then the half X tile
    static constexpr int B_LO = (EXACT ? 2 : 3) * TILE_BYTES;         // offset of B_lo (half: of B_H) inside a stage
    static constexpr int B_H = STD ? 4 * TILE_BYTES : B_LO;
    static constexpr int STAGE_BYTES = HALF ? B_H + HTILE_BYTES : (EXACT ? 3 : 4) * TILE_BYTES;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;
    static constexpr int TMEM_COLS = HALF && EXACT ? 128 : 256;  // main accumulator (+ cross terms)
};
constexpr int B_BOX_BYTES = 32 * BLOCK_K * 4;   // one 32(n) x 32(k) box = 4 KB

constexpr uint32_t IDESC = umma_idesc_tf32(TILE, TILE, /*b_mn_major=*/true);

struct Args {
    int c, hw;
    void* dx;              // float or T
    const float* scale;    // [batch] factor applied in the epilogue, or NULL (= 1)
    const float* mean;     // STD only: [batch * c] per-plane statistics, and the mask [batch, hw] or NULL
    const float* sd;
    const float* mask;
};

template <bool EXACT, typename T, bool STD = false>
__global__ void __launch_bounds__(THREADS, EXACT ? 2 : 1)
isw_sx_tc_kernel(const __grid_constant__ CUtensorMap map_s, const __grid_constant__ CUtensorMap map_x, const Args a) {
    constexpr bool HALF = Cfg<EXACT, T, STD>::HALF;
    constexpr int STAGES = Cfg<EXACT, T, STD>::STAGES, STAGE_BYTES = Cfg<EXACT, T, STD>::STAGE_BYTES;
    constexpr int B_LO = Cfg<EXACT, T, STD>::B_LO;
    constexpr int B_H = Cfg<EXACT, T, STD>::B_H, TMEM_COLS = Cfg<EXACT, T, STD>::TMEM_COLS;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t bars = base + STAGES * STAGE_BYTES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(base_ptr + STAGES * STAGE_BYTES + 8 * (3 * STAGES + 1));
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto ready_bar = [&](int s) { return bars + 8u * (STAGES + s); };
    auto empty_bar = [&](int s) { return bars + 8u * (2 * STAGES + s); };
    const uint32_t accum_bar = bars + 8u * (3 * STAGES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * TILE, m0 = blockIdx.y * TILE, b = blockIdx.z;
    const int n_kb = (a.c + BLOCK_K - 1) / BLOCK_K;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(ready_bar(s), CONVERTER_WARPS);
            mbar_init(empty_bar(s), 1);
        }
        mbar_init(accum_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer: S tile 128(m) x 32(k); X tile 32(k) x 128(n) as four 32-wide n boxes =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_s) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
            for (int kb = 0; kb < n_kb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(empty_bar(s), ph ^ 1u);
                const uint32_t stage = base + s * STAGE_BYTES;
                mbar_arrive_expect_tx(full_bar(s), TILE_BYTES + (HALF ? HTILE_BYTES : TILE_BYTES));
                tma_load_3d(stage, &map_s, full_bar(s), kb * BLOCK_K, m0, b);
                if constexpr (HALF) {
                    tma_load_3d(stage + B_H, &map_x, full_bar(s), n0, kb * BLOCK_K, b);
                } else {
#pragma unroll
                    for (int j = 0; j < TILE / 32; ++j)
                        tma_load_3d(stage + TILE_BYTES + j * B_BOX_BYTES, &map_x, full_bar(s), n0 + 32 * j, kb * BLOCK_K, b);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            for (int kb = 0; kb < n_kb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                if (EXACT) mbar_wait(full_bar(s), ph);  // A goes from TMA straight to the tensor core: observe its arrival here too
                mbar_wait(ready_bar(s), ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t stage = base + s * STAGE_BYTES;
#pragma unroll
                for (int ks = 0; ks < BLOCK_K / UMMA_K; ++ks) {
                    // A (K-major): +32 B inside the swizzle row per k step; B (MN-major): next 8-row k group
                    const uint64_t a_hi = umma_desc_sw128(stage + ks * UMMA_K * 4, 16, 1024);
                    const uint64_t b_hi = umma_desc(stage + TILE_BYTES + ks * 1024, B_BOX_BYTES, 512, 1);
                    if constexpr (HALF && !STD) {  // X_lo == 0
                        umma_tf32(tmem_d, a_hi, b_hi, IDESC, (kb | ks) != 0);
                        if (!EXACT) {
                            const uint64_t a_lo = umma_desc_sw128(stage + 2 * TILE_BYTES + ks * UMMA_K * 4, 16, 1024);
                            umma_tf32(tmem_d + TILE, a_lo, b_hi, IDESC, (kb | ks) != 0);
                        }
                        continue;
                    }
                    const uint64_t b_lo = umma_desc(stage + B_LO + ks * 1024, B_BOX_BYTES, 512, 1);
                    umma_tf32(tmem_d, a_hi, b_hi, IDESC, (kb | ks) != 0);
                    umma_tf32(tmem_d + TILE, a_hi, b_lo, IDESC, (kb | ks) != 0);
                    if (!EXACT) {
                        const uint64_t a_lo = umma_desc_sw128(stage + 2 * TILE_BYTES + ks * UMMA_K * 4, 16, 1024);
                        umma_tf32(tmem_d + TILE, a_lo, b_hi, IDESC, 1u);
                    }
                }
                umma_commit(empty_bar(s));
            }
            umma_commit(accum_bar);
        }
    } else {
        // ===== converters: operand tiles -> hi in place, lo beside (EXACT: only B, A is exact as it is) =====
        const int ctid = threadIdx.x - 64;
        for (int kb = 0; kb < n_kb; ++kb) {
            const int s = kb % STAGES;
            const uint32_t ph = (kb / STAGES) & 1;
            mbar_wait(full_bar(s), ph);
            uint8_t* stage = base_ptr + s * STAGE_BYTES;
            if constexpr (STD) {
                {  // A_lo beside A_hi, as the fp32 general kernel
                    const float4* hi = reinterpret_cast<const float4*>(stage);
                    float4* lo = reinterpret_cast<float4*>(stage + 2 * TILE_BYTES);
#pragma unroll 4
                    for (int i = ctid; i < TILE_BYTES / 16; i += 128) {
                        const float4 v = hi[i];
                        lo[i] = make_float4(tf32_round(v.x - tf32_trunc(v.x)), tf32_round(v.y - tf32_trunc(v.y)),
                                            tf32_round(v.z - tf32_trunc(v.z)), tf32_round(v.w - tf32_trunc(v.w)));
                    }
                }
                // standardise X: this thread's four n values are the same in every k block (n4 = ctid % 32), so is their mask
                const T* src = reinterpret_cast<const T*>(stage + B_H);
                const int n4 = ctid & 31, n = n0 + 4 * n4;
                const bool n_ok = n < a.hw;  // hw % 4 == 0: all four inside or all outside
                float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
                if (a.mask && n_ok) {
                    DGVCC_DEV_CHECK((size_t)b * a.hw + n + 3 < (size_t)gridDim.z * a.hw);
                    const float* mr = a.mask + (size_t)b * a.hw + n;
                    m = make_float4(mr[0], mr[1], mr[2], mr[3]);
                }
#pragma unroll 4
                for (int i = ctid; i < BLOCK_K * TILE / 4; i += 128) {
                    const int kk = i >> 5, ch = kb * BLOCK_K + kk;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (n_ok && ch < a.c) {
                        const size_t si = (size_t)b * a.c + ch;
                        DGVCC_DEV_CHECK(si < (size_t)gridDim.z * a.c);
                        const float mu = a.mean[si], sd = a.sd[si];
                        const float4 xv = widen4(src + kk * TILE + 4 * n4);
                        v.x = __fdiv_rn(__fsub_rn(xv.x, mu), sd);
                        v.y = __fdiv_rn(__fsub_rn(xv.y, mu), sd);
                        v.z = __fdiv_rn(__fsub_rn(xv.z, mu), sd);
                        v.w = __fdiv_rn(__fsub_rn(xv.w, mu), sd);
                        if (a.mask) {
                            v.x = __fmul_rn(v.x, m.x);
                            v.y = __fmul_rn(v.y, m.y);
                            v.z = __fmul_rn(v.z, m.z);
                            v.w = __fmul_rn(v.w, m.w);
                        }
                    }
                    uint8_t* dst = stage + TILE_BYTES + (n4 >> 3) * B_BOX_BYTES + kk * 128 + ((((n4 >> 1) & 3) ^ (kk & 3)) << 5) +
                                   ((n4 & 1) << 4);
                    *reinterpret_cast<float4*>(dst) = v;
                    *reinterpret_cast<float4*>(dst + (B_LO - TILE_BYTES)) =
                        make_float4(tf32_round(v.x - tf32_trunc(v.x)), tf32_round(v.y - tf32_trunc(v.y)),
                                    tf32_round(v.z - tf32_trunc(v.z)), tf32_round(v.w - tf32_trunc(v.w)));
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(ready_bar(s));
                continue;
            } else if constexpr (HALF) {
                if (!EXACT) {  // A_lo beside A_hi
                    const float4* hi = reinterpret_cast<const float4*>(stage);
                    float4* lo = reinterpret_cast<float4*>(stage + 2 * TILE_BYTES);
#pragma unroll 4
                    for (int i = ctid; i < TILE_BYTES / 16; i += 128) {
                        const float4 v = hi[i];
                        lo[i] = make_float4(tf32_round(v.x - tf32_trunc(v.x)), tf32_round(v.y - tf32_trunc(v.y)),
                                            tf32_round(v.z - tf32_trunc(v.z)), tf32_round(v.w - tf32_trunc(v.w)));
                    }
                }
                // widen X: four n values per thread and step; 8 threads fill one 128-byte k row of one box
                const T* src = reinterpret_cast<const T*>(stage + B_H);
#pragma unroll 4
                for (int i = ctid; i < BLOCK_K * TILE / 4; i += 128) {
                    const int kk = i >> 5, n4 = i & 31;
                    uint8_t* dst = stage + TILE_BYTES + (n4 >> 3) * B_BOX_BYTES + kk * 128 + ((((n4 >> 1) & 3) ^ (kk & 3)) << 5) +
                                   ((n4 & 1) << 4);
                    *reinterpret_cast<float4*>(dst) = widen4(src + kk * TILE + 4 * n4);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(ready_bar(s));
                continue;
            }
            // general: [A_hi, B_hi] contiguous -> [A_lo, B_lo] two tiles further; EXACT: B_hi -> B_lo one tile further
            float4* hi = reinterpret_cast<float4*>(stage + (EXACT ? TILE_BYTES : 0));
            float4* lo = reinterpret_cast<float4*>(stage + 2 * TILE_BYTES);
#pragma unroll 4
            for (int i = ctid; i < (EXACT ? 1 : 2) * TILE_BYTES / 16; i += 128) {
                // the tensor core reads only the top 19 bits of a TF32 operand: the raw tile already is hi = trunc(x),
                // only lo = RN_tf32(x - trunc(x)) is written (isw_gram_tc.cu)
                const float4 v = hi[i];
                float4 l;
                l.x = tf32_round(v.x - tf32_trunc(v.x));
                l.y = tf32_round(v.y - tf32_trunc(v.y));
                l.z = tf32_round(v.z - tf32_trunc(v.z));
                l.w = tf32_round(v.w - tf32_trunc(v.w));
                lo[i] = l;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(ready_bar(s));
        }
        // ===== epilogue: TMEM -> dX tile =====
        mbar_wait(accum_bar, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int lane_base = 32 * (warp & 3);
        const int row = m0 + lane_base + lane;
        if constexpr (HALF && !STD) {
            T* out = static_cast<T*>(a.dx) + ((size_t)b * a.c + row) * a.hw + n0;
            const float sc = a.scale ? a.scale[b] : 1.f;
#pragma unroll 1
            for (int c0 = 0; c0 < TILE; c0 += 32) {
                uint32_t r[32], x[32];
                const uint32_t taddr = tmem_d + ((uint32_t)lane_base << 16) + (uint32_t)c0;
                tmem_ld32(taddr, r);
                if (!EXACT) tmem_ld32(taddr + TILE, x);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (row < a.c) {
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const int n = n0 + c0 + 4 * q;
                        if (n >= a.hw) continue;  // hw % 8 == 0: four values are either all inside or all outside
                        float v[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            v[e] = EXACT ? sc * __uint_as_float(r[4 * q + e])
                                         : sc * (__uint_as_float(r[4 * q + e]) + __uint_as_float(x[4 * q + e]));
                        narrow4(out + c0 + 4 * q, v[0], v[1], v[2], v[3]);
                    }
                }
            }
        } else {
        float* out = static_cast<float*>(a.dx) + ((size_t)b * a.c + row) * a.hw + n0;
        const float sc = a.scale ? a.scale[b] : 1.f;
#pragma unroll 1
        for (int c0 = 0; c0 < TILE; c0 += 32) {
            uint32_t r[32], x[32];
            const uint32_t taddr = tmem_d + ((uint32_t)lane_base << 16) + (uint32_t)c0;
            tmem_ld32(taddr, r);
            tmem_ld32(taddr + TILE, x);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (row < a.c) {
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int n = n0 + c0 + 4 * q;
                    if (n < a.hw)  // hw % 4 == 0, so a float4 is either fully inside or fully outside
                        *reinterpret_cast<float4*>(out + c0 + 4 * q) =
                            make_float4(sc * (__uint_as_float(r[4 * q]) + __uint_as_float(x[4 * q])),
                                        sc * (__uint_as_float(r[4 * q + 1]) + __uint_as_float(x[4 * q + 1])),
                                        sc * (__uint_as_float(r[4 * q + 2]) + __uint_as_float(x[4 * q + 2])),
                                        sc * (__uint_as_float(r[4 * q + 3]) + __uint_as_float(x[4 * q + 3])));
                }
            }
        }
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "n"(TMEM_COLS) : "memory");
    }
}

}  // namespace isw_sx
}  // namespace dgvcc

using namespace dgvcc;
using namespace dgvcc::isw_sx;

// fp32 X: four 32(n) x 32(k) boxes per k block in the SWIZZLE_128B_BASE32B layout.  Half X: one raw 32(k) x 128(n) box,
// which the converters widen.
template <typename T, bool STD>
int dgvcc::isw_sx::launch(const float* s, const T* x, const float* mean, const float* sd, const float* mask, int batch, int c,
                          int hw, void* dx, const float* scale, bool exact, cudaStream_t stream) {
    constexpr bool HALF = Cfg<false, T, STD>::HALF;
    if (!(HALF ? half_tc_tiles(c, hw) : sx_tc_tiles(c, hw)) || !tma_aligned(s, x, dx)) return DGVCC_ERR_UNSUPPORTED;
    CUtensorMap map_s, map_x;
    if (!make_tmap_f32_3d(&map_s, s, (uint64_t)c, (uint64_t)c, (uint64_t)batch, TILE)) return DGVCC_ERR_UNSUPPORTED;
    bool mapped;
    if constexpr (HALF)
        mapped = make_tmap_3d(&map_x, HalfIn<T>::TMA, 2, x, (uint64_t)hw, (uint64_t)c, (uint64_t)batch, TILE, BLOCK_K,
                              CU_TENSOR_MAP_SWIZZLE_NONE, 1);
    else
        mapped = make_tmap_f32_3d(&map_x, x, (uint64_t)hw, (uint64_t)c, (uint64_t)batch, BLOCK_K,
                                  CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
    if (!mapped) return DGVCC_ERR_UNSUPPORTED;
    static PerDeviceOnce once;
    if (once.first()) {
        DGVCC_RETURN_IF_CUDA(cudaFuncSetAttribute(isw_sx_tc_kernel<false, T, STD>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                  Cfg<false, T, STD>::SMEM_BYTES));
        if constexpr (!STD)  // STD has no EXACT variant
            DGVCC_RETURN_IF_CUDA(cudaFuncSetAttribute(isw_sx_tc_kernel<true, T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                      Cfg<true, T>::SMEM_BYTES));
    }
    Args a;
    a.c = c; a.hw = hw; a.dx = dx; a.scale = scale;
    a.mean = mean; a.sd = sd; a.mask = mask;
    const dim3 grid(ceil_div(hw, TILE), ceil_div(c, TILE), batch);
    if constexpr (!STD) {
        if (exact) {
            isw_sx_tc_kernel<true, T><<<grid, THREADS, Cfg<true, T>::SMEM_BYTES, stream>>>(map_s, map_x, a);
            return (int)cudaGetLastError();
        }
    }
    isw_sx_tc_kernel<false, T, STD><<<grid, THREADS, Cfg<false, T, STD>::SMEM_BYTES, stream>>>(map_s, map_x, a);
    return (int)cudaGetLastError();
}

template int dgvcc::isw_sx::launch<float, false>(const float*, const float*, const float*, const float*, const float*, int, int,
                                                 int, void*, const float*, bool, cudaStream_t);
template int dgvcc::isw_sx::launch<__half, true>(const float*, const __half*, const float*, const float*, const float*, int, int,
                                                 int, void*, const float*, bool, cudaStream_t);
template int dgvcc::isw_sx::launch<__nv_bfloat16, true>(const float*, const __nv_bfloat16*, const float*, const float*,
                                                        const float*, int, int, int, void*, const float*, bool, cudaStream_t);
template int dgvcc::isw_sx::launch<__half, false>(const float*, const __half*, const float*, const float*, const float*, int,
                                                  int, int, void*, const float*, bool, cudaStream_t);
template int dgvcc::isw_sx::launch<__nv_bfloat16, false>(const float*, const __nv_bfloat16*, const float*, const float*,
                                                         const float*, int, int, int, void*, const float*, bool, cudaStream_t);

extern "C" int dgvcc_isw_sx_tc(const float* s, const float* x, int batch, int c, int hw, float* dx, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!s || !x || !dx || batch <= 0 || c <= 0 || hw <= 0) return DGVCC_ERR_ARG;
    return launch(s, x, nullptr, nullptr, nullptr, batch, c, hw, dx, nullptr, false, (cudaStream_t)stream);
}
