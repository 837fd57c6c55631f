// ISW channel-covariance Gram  G_b = X_b X_b^T  on the Blackwell tensor cores (tcgen05 + TMEM + TMA).
//
// Replaces the torch.bmm of models/ISW/instance_whitening.py:37.  X_b is [C, HW] fp32 with HW
// contiguous, i.e. both MMA operands are K-major.  fp32 accuracy (rtol 1e-5 against the reference's
// sgemm) comes from the 3xTF32 split  x = hi + lo,  hi = RN_tf32(x), lo = RN_tf32(x - hi):
//     G ~= hi hi^T + (hi lo^T + lo hi^T)        (fp32 accumulation in TMEM; lo lo^T ~ 2^-22 is dropped)
// The tensor core truncates (does not round) when it adds into the TMEM accumulator, a bias that grows
// with the number of accumulation steps (measured: -4e-8 relative per K=8 step,
// scripts/probe_tc_accuracy.py).  So (i) the 2^-11-sized cross terms get their own accumulator and
// (ii) a CTA accumulates at most SEG_KB k blocks (64 steps) in TMEM: segments alternate between two
// accumulator sets (TMEM 4 x 128 columns), the epilogue warps drain a finished set into fp32 registers
// (round-to-nearest adds) while the MMAs of the next segment run into the other set.
// One CTA computes one upper-triangular 128x128 tile of one sample over one split of the K = HW range
// and stores the partial tile; isw_cov_finish_kernel (isw_kernels.cu) adds the splits in order.
// C <= 64: the 128-row tile holds TWO samples (TMA box 32 k x 64 rows x 2 samples); their two diagonal
// 64x64 blocks are the Grams, the cross-sample blocks are discarded (50 % useful MMA work instead of 25 %).
//
// Warp roles (320 threads):
//   warp 0   : TMA producer -- cp.async.bulk.tensor of the 128 x 32 fp32 operand tiles (128B swizzle)
//   warp 1   : TMEM allocation; one lane issues tcgen05.mma.kind::tf32 (12 per 32-wide k block)
//   warps 2-9: converters -- write lo beside each landed tile (the tile itself serves as hi), then signal the
//              MMA warp; they also drain finished accumulator sets (tcgen05.ld; warp w reads TMEM lane
//              quarter w % 4, warps 2-5 the left 64 columns, warps 6-9 the right 64) and store the tile
// Pipeline: full[s] (TMA -> converters), ready[s] (converters -> MMA), empty[s] (MMA -> TMA) over
// STAGES shared-memory stages; acc_full[set] (MMA -> drain), acc_empty[set] (drain -> MMA).
//
// Half-precision input (isw_gram_tc_kernel<__half / __nv_bfloat16>): TMA loads the 32 k x 128 row half tiles (64-byte
// rows, no swizzle) behind the two fp32 tiles of the stage, and the converters widen them into those fp32 tiles in the
// 128B-swizzled layout TMA writes for fp32 input.  A widened half value is its own TF32 hi and its lo is exactly 0, so
// the cross accumulator is dropped: one MMA per k step, TMEM 2 x 128 columns, same enable flags, SEG_KB segments and
// drain order, hence the same partials bit for bit as the fp32 kernel on the upcast map.
//
// Standardise on load (isw_gram_tc_kernel<half, STD = true>, the Gram of lw_loss): TMA loads the half x tile as above, and
// the converters compute  v = (x - mean_r) / sd_r  (times mask[sample, k] under a mask) with the IEEE operations of
// lw_standardize_fwd_kernel, write v into the swizzled fp32 hi tile and  lo = RN_tf32(v - trunc_tf32(v))  beside it.  v has
// low bits, so this variant keeps the fp32 kernel's 3 MMAs per k step, its cross accumulator and drains: the tensor core
// sees exactly the operands the fp32 kernel sees on the materialised standardised map, and the partials are the same bits.
// Where TMA zero-fills (k >= hw, rows past C, the missing second sample of an odd pair) the fp32 kernel reads y = 0, so the
// converters write 0 there and read no statistics.  A stage (4 fp32 tiles + 2 half tiles = 80 KB) allows two stages.
#include <type_traits>

#include "isw_tc.cuh"
#include "tc_common.cuh"
#include "../../include/dgvcc_b200.h"

namespace dgvcc {
namespace isw_tc {

constexpr int TILE_M = 128;                 // rows of X per operand tile (= UMMA M = UMMA N)
constexpr int BLOCK_K = 32;                 // fp32 per k block = one 128-byte swizzle row
constexpr int UMMA_K = 8;                   // tf32 MMA k extent (32 bytes)
constexpr bool HI_BY_TRUNCATION = true;     // hi = what the tensor core reads of the raw tile (see the converter loop)
constexpr int SEG_KB = 16;                  // k blocks accumulated in TMEM before a drain (512 k = 64 steps)
constexpr int TILE_BYTES = TILE_M * BLOCK_K * 4;  // 16 KB
constexpr int HTILE_BYTES = TILE_M * BLOCK_K * 2; // 8 KB: a half-precision tile as TMA delivers it
constexpr int CONVERTER_WARPS = 8;                // two per SM sub-partition
constexpr int THREADS = 64 + 32 * CONVERTER_WARPS;
template <typename T, bool STD = false> struct Cfg {
    static constexpr bool HALF = !std::is_same<T, float>::value;
    static constexpr bool LO = !HALF || STD;  // operands with a nonzero TF32 lo part: 3 MMAs per k step, cross accumulator
    static constexpr int STAGES = STD ? 2 : 3;
    // fp32: A_hi, B_hi, A_lo, B_lo.  half: A, B (fp32, widened), then the two half tiles TMA wrote.  STD: A_hi, B_hi, A_lo,
    // B_lo, then the two half tiles
    static constexpr int H_OFF = (LO ? 4 : 2) * TILE_BYTES;  // offset of the half tiles inside a stage
    static constexpr int STAGE_BYTES = HALF ? H_OFF + 2 * HTILE_BYTES : 4 * TILE_BYTES;
    // two accumulator sets, each: hi*hi^T (128 columns) + cross terms (128 columns; none for widened half input)
    static constexpr int TMEM_COLS = LO ? 512 : 256;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*alignment slack*/ + 256 /*barriers*/ +
                                      (STD ? 2 * 2 * TILE_M * 4 : 0) /*mean, sd of the 256 rows*/;
};

using namespace dgvcc::tc;

// K-major operand tiles: rows of 128 B, 8-row swizzle atoms 1024 B apart (SBO); LBO is unused (=16 B).
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) { return umma_desc_sw128(smem_addr, 16, 1024); }

// kind::tf32, fp32 accumulate, A and B K-major, M = N = 128.
constexpr uint32_t IDESC = umma_idesc_tf32(TILE_M, TILE_M, false);

struct Args {
    int c, hw, batch, splits, k_per_split, tiles_1d, n_tiles;
    int pair;     // c <= 64: one CTA holds two samples (64 rows each) in its 128-row tile
    float* part;  // [batch][splits][n_tiles][tile][tile], tile = 64 in pair mode, else 128
    const float* mean;  // STD only: [batch * c] per-plane statistics, and the mask [batch, hw] or NULL
    const float* sd;
    const float* mask;
};

template <typename T, bool STD = false>
__global__ void __launch_bounds__(THREADS, 1)
isw_gram_tc_kernel(const __grid_constant__ CUtensorMap tmap, const Args a) {
    constexpr bool HALF = Cfg<T, STD>::HALF, LO = Cfg<T, STD>::LO;
    constexpr int STAGES = Cfg<T, STD>::STAGES, STAGE_BYTES = Cfg<T, STD>::STAGE_BYTES, TMEM_COLS = Cfg<T, STD>::TMEM_COLS;
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment for the 128B-swizzled tiles
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t bars = base + STAGES * STAGE_BYTES;  // full[S], ready[S], empty[S], acc_full[2], acc_empty[2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(base_ptr + STAGES * STAGE_BYTES + 8 * (3 * STAGES + 4));
    auto full_bar = [&](int s) { return bars + 8u * s; };
    auto ready_bar = [&](int s) { return bars + 8u * (STAGES + s); };
    auto empty_bar = [&](int s) { return bars + 8u * (2 * STAGES + s); };
    auto acc_full_bar = [&](int set) { return bars + 8u * (3 * STAGES + set); };
    auto acc_empty_bar = [&](int set) { return bars + 8u * (3 * STAGES + 2 + set); };

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int ti = 0, rem = blockIdx.x;
    while (rem >= a.tiles_1d - ti) { rem -= a.tiles_1d - ti; ++ti; }
    const int tj = ti + rem;
    const bool diag = ti == tj;  // always true in pair mode (a single tile)
    const int split = blockIdx.y;
    const int b = a.pair ? 2 * blockIdx.z : blockIdx.z;  // first sample of the pair / the sample
    const int k0 = split * a.k_per_split;
    const int k1 = min(a.hw, k0 + a.k_per_split);
    const int n_kb = (k1 - k0 + BLOCK_K - 1) / BLOCK_K;
    const int n_seg = (n_kb + SEG_KB - 1) / SEG_KB;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(ready_bar(s), CONVERTER_WARPS);
            mbar_init(empty_bar(s), 1);
        }
        for (int set = 0; set < 2; ++set) {
            mbar_init(acc_full_bar(set), 1);
            mbar_init(acc_empty_bar(set), CONVERTER_WARPS);
        }
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
        // ===== TMA producer =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
            for (int kb = 0; kb < n_kb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(empty_bar(s), ph ^ 1u);
                const uint32_t stage = base + s * STAGE_BYTES;
                // pair mode: the box is {32 k, 64 rows, 2 samples} = the same 128-row tile
                if constexpr (HALF) {
                    mbar_arrive_expect_tx(full_bar(s), diag ? HTILE_BYTES : 2 * HTILE_BYTES);
                    const uint32_t h = stage + Cfg<T, STD>::H_OFF;
                    tma_load_3d(h, &tmap, full_bar(s), k0 + kb * BLOCK_K, ti * TILE_M, b);
                    if (!diag) tma_load_3d(h + HTILE_BYTES, &tmap, full_bar(s), k0 + kb * BLOCK_K, tj * TILE_M, b);
                } else {
                    mbar_arrive_expect_tx(full_bar(s), diag ? TILE_BYTES : 2 * TILE_BYTES);
                    tma_load_3d(stage, &tmap, full_bar(s), k0 + kb * BLOCK_K, ti * TILE_M, b);
                    if (!diag) tma_load_3d(stage + TILE_BYTES, &tmap, full_bar(s), k0 + kb * BLOCK_K, tj * TILE_M, b);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: segments of SEG_KB k blocks alternate between the two accumulator sets =====
        if (lane == 0) {
            for (int kb = 0; kb < n_kb; ++kb) {
                const int seg = kb / SEG_KB, kin = kb % SEG_KB, set = seg & 1;
                if (kin == 0) {  // the set must have been drained by the epilogue warps (first use passes at once)
                    mbar_wait(acc_empty_bar(set), ((uint32_t)(seg >> 1) & 1u) ^ 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(ready_bar(s), ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t stage = base + s * STAGE_BYTES;
                const uint64_t a_hi = umma_desc(stage);
                const uint64_t b_hi = umma_desc(stage + (diag ? 0 : TILE_BYTES));
                if constexpr (!LO) {  // lo == 0: hi hi^T only
                    const uint32_t d_main = tmem_d + (uint32_t)set * TILE_M;
#pragma unroll
                    for (int ks = 0; ks < BLOCK_K / UMMA_K; ++ks) {
                        const uint64_t adv = (uint64_t)((ks * UMMA_K * 4) >> 4);
                        umma_tf32(d_main, a_hi + adv, b_hi + adv, IDESC, (kin | ks) != 0);
                    }
                } else {
                    const uint64_t a_lo = umma_desc(stage + 2 * TILE_BYTES);
                    const uint64_t b_lo = umma_desc(stage + (diag ? 2 : 3) * TILE_BYTES);
                    const uint32_t d_main = tmem_d + (uint32_t)set * 2 * TILE_M, d_cross = d_main + TILE_M;
#pragma unroll
                    for (int ks = 0; ks < BLOCK_K / UMMA_K; ++ks) {
                        const uint64_t adv = (uint64_t)((ks * UMMA_K * 4) >> 4);  // +32 B inside the swizzle row
                        umma_tf32(d_main, a_hi + adv, b_hi + adv, IDESC, (kin | ks) != 0);
                        umma_tf32(d_cross, a_hi + adv, b_lo + adv, IDESC, (kin | ks) != 0);
                        umma_tf32(d_cross, a_lo + adv, b_hi + adv, IDESC, 1u);
                    }
                }
                umma_commit(empty_bar(s));  // frees the stage once these MMAs have read it
                if (kin == SEG_KB - 1 || kb == n_kb - 1) umma_commit(acc_full_bar(set));
            }
        }
    } else {
        // ===== converters (lo beside the tile; hi = the tile as delivered) and, lagging two k blocks behind, the segment drains =====
        const int ctid = threadIdx.x - 64;      // 0..255
        const int lane_base = 32 * (warp & 3);  // a warp may only touch its own quarter of the TMEM lanes
        const int row = lane_base + lane;       // row of the 128 x 128 tile held by this thread
        const int col_begin = (warp - 2) / 4 * (TILE_M / 2);  // warps 2-5: columns 0-63, warps 6-9: 64-127
        // pair mode: rows 0-63 x columns 0-63 is sample b, rows 64-127 x columns 64-127 is sample b+1; the
        // other two quadrants are cross-sample products nobody needs
        const bool useful = !a.pair || (row >> 6) == (col_begin >> 6);
        float acc[TILE_M / 2];
#pragma unroll
        for (int q = 0; q < TILE_M / 2; ++q) acc[q] = 0.f;

        auto drain = [&](int seg) {
            const int set = seg & 1;
            mbar_wait(acc_full_bar(set), (uint32_t)(seg >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if constexpr (!LO) {
                if (useful) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        uint32_t r[32];
                        tmem_ld32(tmem_d + ((uint32_t)lane_base << 16) + (uint32_t)(set * TILE_M + col_begin + 32 * h), r);
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int q = 0; q < 32; ++q) acc[32 * h + q] += __uint_as_float(r[q]);
                    }
                }
            } else if (useful) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    uint32_t r[32], x[32];
                    const uint32_t taddr = tmem_d + ((uint32_t)lane_base << 16) + (uint32_t)(set * 2 * TILE_M + col_begin + 32 * h);
                    tmem_ld32(taddr, r);           // hi hi^T
                    tmem_ld32(taddr + TILE_M, x);  // hi lo^T + lo hi^T
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int q = 0; q < 32; ++q) acc[32 * h + q] += __uint_as_float(r[q]) + __uint_as_float(x[q]);
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty_bar(set));
        };

        // STD: the statistics of the tile's 256 rows (A then B) go to shared memory once, thread ctid loading row ctid.
        // This thread converts k chunk k4 of rows rr = ctid / 8 + 32 j (j < 4 on a diagonal tile) in every k block; a row
        // that does not exist (past C, or the missing sample of an odd pair) has its bit of ok clear and is written as 0,
        // like the rows TMA zero-fills for the fp32 kernel, and no statistics are read for it.
        float* s_mu = reinterpret_cast<float*>(base_ptr + STAGES * STAGE_BYTES + 256);
        float* s_sd = s_mu + 2 * TILE_M;
        uint32_t ok = 0;
        if constexpr (STD) {
            auto row_of = [&](int rr, size_t& si) {  // false when row rr of [A; B] does not exist; else si = its plane
                const int r = rr & (TILE_M - 1);
                int sample, ch;
                if (a.pair) { sample = b + (r >> 6); ch = r & 63; }
                else { sample = b; ch = (rr < TILE_M ? ti : tj) * TILE_M + r; }
                si = (size_t)sample * a.c + ch;
                return sample < a.batch && ch < a.c && (rr < TILE_M || !diag);
            };
            size_t si;
            if (row_of(ctid, si)) {
                DGVCC_DEV_CHECK(si < (size_t)a.batch * a.c);
                s_mu[ctid] = a.mean[si];
                s_sd[ctid] = a.sd[si];
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (row_of((ctid >> 3) + 32 * j, si)) ok |= 1u << j;
            asm volatile("bar.sync 1, %0;" ::"n"(32 * CONVERTER_WARPS) : "memory");  // the converter warps only
        }

        int drained = 0;
        for (int kb = 0; kb < n_kb; ++kb) {
            const int s = kb % STAGES;
            const uint32_t ph = (kb / STAGES) & 1;
            mbar_wait(full_bar(s), ph);
            uint8_t* stage = base_ptr + s * STAGE_BYTES;
            if constexpr (STD) {
                const T* src = reinterpret_cast<const T*>(stage + Cfg<T, STD>::H_OFF);
                const int k4 = ctid & 7, kg = k0 + kb * BLOCK_K + 4 * k4;
                const bool k_ok = kg < a.hw;  // hw % 4 == 0: the four k values are all inside or all outside
                // mask values of the (at most two) samples of this tile at k = kg..kg+3
                float4 m0 = make_float4(1.f, 1.f, 1.f, 1.f), m1 = m0;
                if (a.mask && k_ok) {
                    DGVCC_DEV_CHECK((size_t)b * a.hw + kg + 3 < (size_t)a.batch * a.hw);
                    const float* mr = a.mask + (size_t)b * a.hw + kg;
                    m0 = make_float4(mr[0], mr[1], mr[2], mr[3]);
                    if (a.pair && b + 1 < a.batch) {
                        mr += a.hw;
                        m1 = make_float4(mr[0], mr[1], mr[2], mr[3]);
                    }
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (j >= 4 && diag) break;
                    const int rr = (ctid >> 3) + 32 * j;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (k_ok && (ok >> j & 1u)) {
                        // the operations of lw_standardize_fwd_kernel: (x - mean) / sd, then * mask
                        const float4 xv = widen4(src + rr * BLOCK_K + 4 * k4);
                        const float mu = s_mu[rr], sd = s_sd[rr];
                        v.x = __fdiv_rn(__fsub_rn(xv.x, mu), sd);
                        v.y = __fdiv_rn(__fsub_rn(xv.y, mu), sd);
                        v.z = __fdiv_rn(__fsub_rn(xv.z, mu), sd);
                        v.w = __fdiv_rn(__fsub_rn(xv.w, mu), sd);
                        if (a.mask) {
                            const float4 m = a.pair && (rr & (TILE_M - 1)) >= 64 ? m1 : m0;
                            v.x = __fmul_rn(v.x, m.x);
                            v.y = __fmul_rn(v.y, m.y);
                            v.z = __fmul_rn(v.z, m.z);
                            v.w = __fmul_rn(v.w, m.w);
                        }
                    }
                    // hi = v as the tensor core truncates it, lo = RN_tf32(v - trunc(v)) at the same swizzled place
                    const int off = rr * 128 + ((k4 ^ (rr & 7)) << 4);
                    *reinterpret_cast<float4*>(stage + off) = v;
                    *reinterpret_cast<float4*>(stage + 2 * TILE_BYTES + off) =
                        make_float4(tf32_round(v.x - tf32_trunc(v.x)), tf32_round(v.y - tf32_trunc(v.y)),
                                    tf32_round(v.z - tf32_trunc(v.z)), tf32_round(v.w - tf32_trunc(v.w)));
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(ready_bar(s));
                while (drained < n_seg - 1 && kb >= (drained + 1) * SEG_KB + 1) drain(drained++);
                continue;
            } else if constexpr (HALF) {
                // widen [A; B] (128 or 256 rows of 32 half values) into the fp32 tiles: one float4 per thread and step,
                // 16-byte chunk k4 of row r at chunk k4 ^ (r % 8) of the 128-byte row (the 128B swizzle)
                const T* src = reinterpret_cast<const T*>(stage + Cfg<T, STD>::H_OFF);
#pragma unroll 4
                for (int i = ctid; i < (diag ? 1 : 2) * TILE_M * (BLOCK_K / 4); i += 32 * CONVERTER_WARPS) {
                    const int r = i >> 3, k4 = i & 7;
                    *reinterpret_cast<float4*>(stage + r * 128 + ((k4 ^ (r & 7)) << 4)) = widen4(src + r * BLOCK_K + 4 * k4);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(ready_bar(s));
                while (drained < n_seg - 1 && kb >= (drained + 1) * SEG_KB + 1) drain(drained++);
                continue;
            }
            const int n_vec = (diag ? 1 : 2) * (TILE_BYTES / 16);  // float4s of A_hi (and B_hi, contiguous after it)
            float4* hi = reinterpret_cast<float4*>(stage);
            float4* lo = reinterpret_cast<float4*>(stage + 2 * TILE_BYTES);
#pragma unroll 4
            for (int i = ctid; i < n_vec; i += 32 * CONVERTER_WARPS) {
                const float4 v = hi[i];
                float4 l;
                if (HI_BY_TRUNCATION) {
                    // the tensor core reads only the top 19 bits of a TF32 operand, so the raw tile IS hi = trunc(x);
                    // only lo = RN_tf32(x - trunc(x)) has to be written
                    l.x = tf32_round(v.x - tf32_trunc(v.x));
                    l.y = tf32_round(v.y - tf32_trunc(v.y));
                    l.z = tf32_round(v.z - tf32_trunc(v.z));
                    l.w = tf32_round(v.w - tf32_trunc(v.w));
                } else {
                    float4 h;
                    h.x = tf32_round(v.x); l.x = tf32_round(v.x - h.x);
                    h.y = tf32_round(v.y); l.y = tf32_round(v.y - h.y);
                    h.z = tf32_round(v.z); l.z = tf32_round(v.z - h.z);
                    h.w = tf32_round(v.w); l.w = tf32_round(v.w - h.w);
                    hi[i] = h;
                }
                lo[i] = l;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic writes -> tensor-core reads
            __syncwarp();
            if (lane == 0) mbar_arrive(ready_bar(s));
            // a finished segment is drained once two k blocks of the next one are converted: by then its MMAs
            // have completed, so the drain does not stall the conversion pipeline
            while (drained < n_seg - 1 && kb >= (drained + 1) * SEG_KB + 1) drain(drained++);
        }
        while (drained < n_seg) drain(drained++);

        // ===== epilogue: register sums -> global partial tile =====
        if (useful) {
            float* out;
            bool row_ok;
            int col_limit;  // valid columns of this thread's 64-column half
            if (a.pair) {
                const int sample = b + (row >> 6), r64 = row & 63;
                out = a.part + ((((size_t)sample * a.splits + split) * 64 + r64) * 64);
                row_ok = sample < a.batch && r64 < a.c;
                col_limit = a.c;
            } else {
                out = a.part + ((((size_t)b * a.splits + split) * a.n_tiles + blockIdx.x) * TILE_M + row) * TILE_M + col_begin;
                row_ok = ti * TILE_M + row < a.c;
                col_limit = a.c - (tj * TILE_M + col_begin);
            }
            if (row_ok) {
#pragma unroll
                for (int q = 0; q < TILE_M / 8; ++q)
                    if (4 * q < col_limit)
                        *reinterpret_cast<float4*>(out + 4 * q) = make_float4(acc[4 * q], acc[4 * q + 1], acc[4 * q + 2], acc[4 * q + 3]);
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

}  // namespace isw_tc
}  // namespace dgvcc

using namespace dgvcc;
using namespace dgvcc::isw_tc;

// fp32 x: the 128B-swizzled tiles the MMAs read.  Half x: its raw 32 k x 128 row tiles, which the converters widen.
template <typename T, bool STD>
int dgvcc::isw_tc::launch(const T* x, const float* mean, const float* sd, const float* mask, int batch, int c, int hw,
                          int splits, int k_per_split, float* part, cudaStream_t stream) {
    constexpr bool HALF = Cfg<T, STD>::HALF;
    // rows past C are zero-filled by the tensor map, so C needs no multiple of the tile
    if (!(HALF ? half_tc_tiles(c, hw) : gram_tc_tiles(c, hw)) || k_per_split % BLOCK_K != 0 || !tma_aligned(x))
        return DGVCC_ERR_UNSUPPORTED;
    const int pair = c <= 64;
    CUtensorMap tmap;
    bool mapped;
    if constexpr (HALF)
        mapped = make_tmap_3d(&tmap, HalfIn<T>::TMA, 2, x, (uint64_t)hw, (uint64_t)c, (uint64_t)batch, BLOCK_K,
                              pair ? 64 : TILE_M, CU_TENSOR_MAP_SWIZZLE_NONE, pair ? 2 : 1);
    else
        mapped = make_tmap_f32_3d(&tmap, x, (uint64_t)hw, (uint64_t)c, (uint64_t)batch, pair ? 64 : TILE_M,
                                  CU_TENSOR_MAP_SWIZZLE_128B, pair ? 2 : 1);
    if (!mapped) return DGVCC_ERR_UNSUPPORTED;
    static PerDeviceOnce once;
    if (once.first())
        DGVCC_RETURN_IF_CUDA(cudaFuncSetAttribute(isw_gram_tc_kernel<T, STD>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                  Cfg<T, STD>::SMEM_BYTES));
    Args a;
    a.c = c; a.hw = hw; a.batch = batch; a.splits = splits; a.k_per_split = k_per_split;
    a.pair = pair;
    a.tiles_1d = pair ? 1 : ceil_div(c, TILE_M);
    a.n_tiles = a.tiles_1d * (a.tiles_1d + 1) / 2;
    a.part = part;
    a.mean = mean; a.sd = sd; a.mask = mask;
    const int grid_z = pair ? ceil_div(batch, 2) : batch;
    isw_gram_tc_kernel<T, STD><<<dim3(a.n_tiles, splits, grid_z), THREADS, Cfg<T, STD>::SMEM_BYTES, stream>>>(tmap, a);
    return (int)cudaGetLastError();
}

template int dgvcc::isw_tc::launch<float, false>(const float*, const float*, const float*, const float*, int, int, int, int,
                                                 int, float*, cudaStream_t);
template int dgvcc::isw_tc::launch<__half, false>(const __half*, const float*, const float*, const float*, int, int, int, int,
                                                  int, float*, cudaStream_t);
template int dgvcc::isw_tc::launch<__nv_bfloat16, false>(const __nv_bfloat16*, const float*, const float*, const float*, int,
                                                         int, int, int, int, float*, cudaStream_t);
template int dgvcc::isw_tc::launch<__half, true>(const __half*, const float*, const float*, const float*, int, int, int, int,
                                                 int, float*, cudaStream_t);
template int dgvcc::isw_tc::launch<__nv_bfloat16, true>(const __nv_bfloat16*, const float*, const float*, const float*, int,
                                                        int, int, int, int, float*, cudaStream_t);

extern "C" int dgvcc_isw_gram_tc_partials(const float* x, int batch, int c, int hw, int splits, int k_per_split,
                                          float* part, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!x || !part || batch <= 0 || c <= 0 || hw <= 0 || splits <= 0 || k_per_split <= 0) return DGVCC_ERR_ARG;
    return launch(x, nullptr, nullptr, nullptr, batch, c, hw, splits, k_per_split, part, (cudaStream_t)stream);
}
