// Fused Bayesian-loss forward/backward for sm_100a.
//
// Replaces losses/bl.py (Post_Prob + Bay_Loss + autograd) of the reference without ever
// materialising the [points x pixels] posterior.  Work decomposition ("pixel owner"):
//   warp task  = (point chunk of one image, block of 32*C grid columns, band of R grid rows);
//                lane <-> grid column (C columns 32 apart per lane), each thread owns R*C pixels in
//                registers;
//   the warp streams the chunk's points through a private shared-memory tile (x, x*x and the R
//   per-row y-distances of each point), so the inner loop per (point, pixel) pair is
//   FADD, FFMA, FMUL, MUFU.EX2, FADD/FFMA.  ncu (profiles/) shows the kernels bound by the SM's MIO
//   path that MUFU shares with LDS/SHFL, which is why each thread owns as many pixels as registers
//   allow: 3 broadcast LDS feed R*C exponentials.
// Launch sequence of one forward + backward (7 launches; dense unless exact_cull is set):
//   K0 bl_grid_build_kernel + bl_gridmin_kernel : per-pixel min_n dis over ALL points of an image (bl.py:39) through a
//                         uniform grid over the points (counting sort per image, ring walk per 2 x 32 pixel tile)
//   K1 bl_z_kernel      : softmax max incl. background row + denominator shares (bl.py:39-44); the last chunk to
//                         arrive at a pixel tile adds the shares in chunk order and writes 1/Z and the bg posterior
//   K2 bl_counts_kernel : expected counts c_n = sum_m D[m] p[n,m]   (bl.py:73), one partial row per CTA of 4 tiles
//   K3 bl_reduce_counts_kernel + bl_select_kernel : deterministic reduction of the partials,
//                         |t-c|, trimmed top-k (radix select), loss (bl.py:75-79)
//   K4 bl_grad_kernel   : dL/dD[m] = g * sum_n w_n p[n,m]            (autograd of bl.py:73-79); last arrival finishes
// K1, K2, K4 are persistent (work queue, longest chunks first).  Big images are cut into near-equal point chunks
// (host-built table) so every warp task costs about the same; per-chunk partial denominators / gradient sums are
// combined in chunk order (deterministic, no float atomics).  The second half of the file holds the two multi-GPU
// variants (point-chunk sharding, row-band sharding): the same kernels with the exchange fused in (struct Xchg).
//
// Rounding contract (SURVEY.md section 0 / Appendix A): the softmax arguments reproduce the
// reference's fp32 sequence bit for bit -- no FMA contraction in the distance expansion
// (explicit _rn intrinsics), IEEE sqrt, IEEE division by 2*sigma^2 (exact scaling when it is
// a power of two, otherwise a Markstein-corrected reciprocal multiply that is correctly
// rounded).  Only exp (one MUFU.EX2 fed by one fused multiply-add, see pair_exp) and the summation order
// differ, ~1e-6.
#include <stdlib.h>
#include <string.h>

#include <mutex>

#include "common.cuh"
#include "../../include/dgvcc_b200.h"

namespace dgvcc {
namespace bl {

constexpr int WARPS_PER_CTA = 4;
constexpr int CTA_THREADS = WARPS_PER_CTA * 32;
constexpr int TILE_PTS = 128;  // points staged per warp per tile
constexpr int COUNT_SPAN = 1024;  // points whose partial counts a CTA combines in shared memory per pass
static_assert(COUNT_SPAN % TILE_PTS == 0 && WARPS_PER_CTA == 4, "bl_counts_kernel's CTA combine");

struct Scale {
    float s;          // fl32(2*sigma^2)                     bl.py:42
    float r;          // RN(1/s)
    float neg_inv_s;  // -1/s (exact when s is a power of two)
    float k1;         // -log2(e)/s: exponent slope per unit of squared distance
};

struct Geom {
    int hp, wp;        // grid rows, columns
    int col_blocks;    // ceil(wp / (32*C))
    int tiles;         // warp tasks per (image, chunk) = col_blocks * ceil(hp / R); a launch sweeps [task_first, tiles)
    int task_first;    // 0, or (row-band sharding) the first warp task of the band of grid rows this rank sweeps
    int tiles_img;     // warp tasks per (image, chunk) over the WHOLE grid (stride of the per-tile arrival counters)
    float stride;      // image pixels per grid cell
    float half;        // stride / 2
};

// -dis / s, rounded exactly like the reference's true division.
template <bool POW2>
__device__ __forceinline__ float neg_div(float dis, const Scale& k) {
    if (POW2) return __fmul_rn(dis, k.neg_inv_s);
    const float x = -dis;
    const float q = __fmul_rn(x, k.r);
    const float rem = __fmaf_rn(-q, k.s, x);
    return __fmaf_rn(rem, k.r, q);
}

// exp(a - amax) with a = -dis/s, as 2^((a - amax) log2 e) in ONE fused multiply-add feeding MUFU.EX2:
//   power-of-two s : fma(dis, -log2e/s, k2)         general s : fma(RN(-dis/s), log2e, k2)
// with k2 = fl(-amax * log2e) fixed per pixel.  The rounding of k2 (and, for power-of-two s, of the
// slope) moves every exponent of one pixel by the same amount, which cancels in e / sum(e); what is left
// is |t| * 2^-23 per term, the same size as rounding (a - amax) and its product with log2e separately.
// The kernels are instruction-issue bound next to MUFU, so one instruction fewer per pair is ~5 %.
template <bool POW2>
__device__ __forceinline__ float pair_exp(float dis, float k2, const Scale& k) {
    if (POW2) return ex2_ftz(__fmaf_rn(dis, k.k1, k2));
    return ex2_ftz(__fmaf_rn(neg_div<false>(dis, k), LOG2E, k2));
}

// Two fp32 values in one 64-bit register: Blackwell's packed add/mul/fma.f32x2 (SASS FADD2 / FMUL2 / FFMA2)
// do the work of two scalar instructions in one issue slot; each lane is an ordinary IEEE round-to-nearest op.
typedef unsigned long long f2;
__device__ __forceinline__ f2 pack2(float lo, float hi) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(f2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { f2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { f2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

// Broadcast copies of the Scale constants for the packed path.
struct Scale2 {
    f2 k1, neg_s, r, neg_l;
    __device__ __forceinline__ explicit Scale2(const Scale& k)
        : k1(pack2(k.k1, k.k1)), neg_s(pack2(-k.s, -k.s)), r(pack2(k.r, k.r)), neg_l(pack2(-LOG2E, -LOG2E)) {}
};

// pair_exp for two pixels at once (same arithmetic per lane as the scalar version).
template <bool POW2>
__device__ __forceinline__ f2 pair_exp2(f2 dis, f2 k2, const Scale2& k) {
    f2 t;
    if (POW2) {
        t = fma2(dis, k.k1, k2);
    } else {
        // dis / s correctly rounded (Markstein), then t = (-dis/s) * log2e + k2 in one fma
        const f2 q = mul2(dis, k.r);
        const f2 rem = fma2(q, k.neg_s, dis);
        t = fma2(fma2(rem, k.r, q), k.neg_l, k2);
    }
    float t0, t1;
    unpack2(t, t0, t1);
    return pack2(ex2_ftz(t0), ex2_ftz(t1));
}

// ((-2 * fl(p*c)) + fl(p*p)) + fl(c*c)   bl.py:27-28;  cm2 = -2c (scaling by 2 commutes with rounding)
__device__ __forceinline__ float axis_sqdist(float p, float pp, float cm2, float cc) {
    return __fadd_rn(__fadd_rn(__fmul_rn(p, cm2), pp), cc);
}

// Grid-cell centre, bl.py:14-15: arange(0, c_size, stride) + stride/2 (exact for integer strides).
__device__ __forceinline__ float cell_centre(int idx, const Geom& g) {
    return __fadd_rn(__fmul_rn((float)idx, g.stride), g.half);
}

template <int R>
struct __align__(16) WarpTile {
    float2 xs[TILE_PTS];      // (x, x*x)
    float yd[TILE_PTS][R];    // y-axis squared distance to each of the warp's R rows
    float aux[TILE_PTS];      // K2: staged counts; K4: signed weights
    unsigned char idx[TILE_PTS];  // K2 with culling: position of each kept point inside the staged tile
};

// Views into the host-built int32 table (layout documented in include/dgvcc_b200.h).
struct Meta {
    const int32_t* pt_off;   // [B+1]
    const int32_t* row_off;  // [B+1]
    const int32_t* keep;     // [B]
    const int32_t* icb;      // [B+1] first point-chunk id of each image
    const int32_t* chunks;   // [C][4] = (image, first point, point count, chunk id run in launch slot c)
};

__host__ __device__ __forceinline__ Meta meta_view(const int32_t* m, int batch) {
    Meta v;
    v.pt_off = m;
    v.row_off = m + (batch + 1);
    v.keep = m + 2 * (batch + 1);
    v.icb = m + 3 * batch + 2;
    v.chunks = m + 4 * batch + 3;
    return v;
}

// Point-chunk sharding across GPUs (dgvcc_bl_shard_*): this rank owns the chunk ids [chunk_lo, chunk_hi), i.e. the
// points [pt_lo, pt_hi) of the packed sequence, and touches the images [img_lo, img_hi).  One GPU: on = 0.
struct Shard {
    int on;
    int chunk_lo, chunk_hi, pt_lo, pt_hi, img_lo, img_hi;
};
__host__ __device__ __forceinline__ Shard no_shard() { return Shard{0, 0, 0x7fffffff, 0, 0x7fffffff, 0, 0x7fffffff}; }

// Peer exchange of the sharded path, fused into the kernels that produce / consume the data.  A producing kernel
// stores its results into its own workspace AND, with plain stores over NVLink, into the workspaces of the ranks in
// the destination mask of its chunk / image; when its last CTA is done (every CTA fences its remote stores at system
// scope before it takes a ticket) it raises this rank's flag of the phase on the ranks in signal_mask.  A consuming
// kernel first waits for the flags of the ranks in wait_mask (bounded: a lost peer leaves a code in err[0], not a hung
// GPU).  peers == nullptr and wait_mask == 0 (the value-initialised struct): one GPU, nothing happens.
struct Xchg {
    char* const* peers;         // [world] workspace bases as mapped into this process (own one included)
    const unsigned int* mask;   // destination ranks per chunk (sweeps) or per image (row / image kernels)
    unsigned int* ticket;       // CTA arrival counter of the producing kernel (zero between kernels)
    const unsigned int* flags;  // this rank's own flag array [phase][source]
    int* err;
    long long flags_off;        // byte offset of the flag array in every workspace
    long long region_off, region_off2;  // byte offsets of the exchanged arrays in every workspace
    int phase, rank, world;     // producing side: phase raised
    unsigned int signal_mask, epoch;
    unsigned int wait_mask, wait_mask2;  // consuming side: up to two phases to wait for
    int wait_phase, wait_phase2;
};

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
constexpr unsigned long long XCHG_TIMEOUT_NS = 2000000000ull;  // 2 s

__device__ __forceinline__ void xchg_spin(const unsigned int* flag, unsigned int epoch, int code, int* err) {
    const unsigned long long t0 = global_ns();
    while ((int)(ld_acquire_sys(flag) - epoch) < 0) {
        if (global_ns() - t0 > XCHG_TIMEOUT_NS) {
            atomicExch(err, code);
            break;
        }
        __nanosleep(32);
    }
}

// Consumer prologue, called by every thread of the CTA: lane = source rank, warp 0 / 1 = first / second phase.
__device__ __forceinline__ void xchg_wait(const Xchg& x) {
    if ((x.wait_mask | x.wait_mask2) == 0u) return;
    const int src = threadIdx.x & 31, which = threadIdx.x >> 5;
    if (which < 2 && src < x.world) {
        const unsigned int m = which ? x.wait_mask2 : x.wait_mask;
        const int ph = which ? x.wait_phase2 : x.wait_phase;
        if ((m >> src) & 1u) xchg_spin(x.flags + ph * x.world + src, x.epoch, 1 + ph + 16 * src, x.err);
    }
    // the polling threads' ld.acquire.sys + the CTA barrier order every thread's later loads after the peers' stores
    // (causality is transitive over the barrier); a system-scope fence here cost ~5 us per consumer kernel
    __syncthreads();
}

// Base of an exchanged array on rank q.
__device__ __forceinline__ float* xchg_ptr(const Xchg& x, int q, long long region_off) {
    DGVCC_DEV_CHECK(q >= 0 && q < x.world && region_off >= 0);
    return reinterpret_cast<float*>(x.peers[q] + region_off);
}

// One value into the same array of every rank in `mask`.
__device__ __forceinline__ void xchg_store(const Xchg& x, unsigned int mask, long long region_off, size_t elem, float v) {
    while (mask) {
        const int q = __ffs(mask) - 1;
        mask &= mask - 1u;
        DGVCC_DEV_CHECK(q < x.world && region_off >= 0);
        reinterpret_cast<float*>(x.peers[q] + region_off)[elem] = v;
    }
}

// Producer epilogue, called by every thread of every CTA of the grid (no early returns before it).
// `stored`: this thread wrote to a peer (only then does it pay for the system-scope fence; a CTA that kept everything
// at home just takes its ticket).
__device__ __forceinline__ void xchg_signal(const Xchg& x, bool stored = true) {
    if (!x.peers) return;
    // device-scope acq_rel fence per storing thread; the thread that raises the flags acquires them through the ticket
    // and publishes everything with its st.release.sys (release is cumulative) -- no fence.sc.sys on the path
    if (stored) fence_acq_rel_gpu();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int total = gridDim.x * gridDim.y * gridDim.z;
        if (atomicAdd(x.ticket, 1u) == total - 1u) {
            fence_acq_rel_gpu();  // acquires the other CTAs' stores; the st.release.sys below publishes them (cumulative)
            unsigned int m = x.signal_mask;
            while (m) {
                const int q = __ffs(m) - 1;
                m &= m - 1u;
                st_release_sys(reinterpret_cast<unsigned int*>(x.peers[q] + x.flags_off) + x.phase * x.world + x.rank, x.epoch);
            }
            *x.ticket = 0u;
        }
    }
}

struct TaskInfo {
    int img, row0, n_rows;    // image, its first posterior row, number of rows
    int n_img_pts;            // points in the whole image
    int pt_base;              // index of the chunk's first point in the packed arrays
    int p_start, p_cnt;       // chunk = points [p_start, p_start + p_cnt) of the image
    int chunk, first_chunk, n_chunks;
    int col0, row_base;       // this lane's first column, first row of the band
    int task;                 // pixel-tile index inside the image
};

// One warp task = (point chunk, block of 32*C columns, band of R rows).  Chunks are equal-sized slices
// of an image's points so that all tasks cost the same and the hardware CTA scheduler balances them.
template <int R, int C>
__device__ __forceinline__ bool decode_task(const int32_t* __restrict__ meta, int batch, const Geom& g,
                                            TaskInfo& t, int slot, int task) {
    const int lane = threadIdx.x & 31;
    t.task = task;
    const Meta mv = meta_view(meta, batch);
    t.chunk = mv.chunks[4 * slot + 3];
    const int32_t* ce = mv.chunks + 4 * t.chunk;
    t.img = ce[0];
    t.p_start = ce[1];
    t.p_cnt = ce[2];
    t.first_chunk = mv.icb[t.img];
    t.n_chunks = mv.icb[t.img + 1] - t.first_chunk;
    const int pt0 = mv.pt_off[t.img];
    t.n_img_pts = mv.pt_off[t.img + 1] - pt0;
    t.pt_base = pt0 + t.p_start;
    t.row0 = mv.row_off[t.img];
    t.n_rows = mv.row_off[t.img + 1] - t.row0;
    const int jb = t.task % g.col_blocks, kb = t.task / g.col_blocks;
    t.col0 = jb * 32 * C + lane;
    t.row_base = kb * R;
    DGVCC_DEV_CHECK(slot >= 0 && task >= 0 && t.chunk >= 0);
    DGVCC_DEV_CHECK(t.img >= 0 && t.img < batch);
    DGVCC_DEV_CHECK(t.chunk >= t.first_chunk && t.chunk < t.first_chunk + max(t.n_chunks, 1));
    DGVCC_DEV_CHECK(t.p_start >= 0 && t.p_cnt >= 0 && t.p_start + t.p_cnt <= t.n_img_pts);
    DGVCC_DEV_CHECK(t.n_rows >= t.n_img_pts && t.n_rows <= t.n_img_pts + 1 && t.row0 >= 0 && pt0 >= 0);
    DGVCC_DEV_CHECK(t.task >= g.tiles || t.row_base < g.hp);
    return t.task < g.tiles;  // the chunk fields are valid either way (all warps of a CTA share the chunk)
}

// Stage `padded` points starting at pts[n0] (lane-strided, coalesced float2 loads); entries at or
// past `limit` repeat the last valid point so that padding stays finite.
template <int R>
__device__ __forceinline__ void stage_points(WarpTile<R>& tile, const float2* __restrict__ pts, int n0,
                                             int limit, int padded, const float (&cym2)[R],
                                             const float (&cyy)[R]) {
    const int lane = threadIdx.x & 31;
#pragma unroll 1
    for (int i = lane; i < padded; i += 32) {
        const int n = min(n0 + i, limit - 1);
        DGVCC_DEV_CHECK(n >= 0 && i < TILE_PTS);
        const float2 p = __ldg(&pts[n]);
        tile.xs[i] = make_float2(p.x, __fmul_rn(p.x, p.x));
        const float yy = __fmul_rn(p.y, p.y);
#pragma unroll
        for (int r = 0; r < R; ++r) tile.yd[i][r] = axis_sqdist(p.y, yy, cym2[r], cyy[r]);
    }
}

// Same with a per-point predicate keep(x, y, w): only the points it accepts are staged, compacted in
// order (ballot/popc), so sums stay deterministic.  Returns the number kept.  HAS_W: weights w[n0+i]
// are read and land in tile.aux; HAS_IDX: tile.idx[pos] records the point's position in the tile.
template <int R, bool HAS_W, bool HAS_IDX, int UNROLL = 1, typename Keep>
__device__ __forceinline__ int stage_points_if(WarpTile<R>& tile, const float2* __restrict__ pts,
                                               const float* __restrict__ w, int n0, int cnt,
                                               const float (&cym2)[R], const float (&cyy)[R], Keep keep_fn) {
    const int lane = threadIdx.x & 31;
    int kept = 0;
#pragma unroll UNROLL
    for (int base = 0; base < cnt; base += 32) {
        const int i = base + lane;
        float2 p = make_float2(0.f, 0.f);
        float wi = 1.f;
        bool keep = false;
        if (i < cnt) {
            p = __ldg(&pts[n0 + i]);
            if (HAS_W) wi = __ldg(&w[n0 + i]);
            keep = keep_fn(p.x, p.y, wi);
        }
        const unsigned int ballot = __ballot_sync(FULL_MASK, keep);
        if (keep) {
            const int pos = kept + __popc(ballot & ((1u << lane) - 1u));
            DGVCC_DEV_CHECK(pos >= 0 && pos < TILE_PTS && n0 + i >= 0);
            tile.xs[pos] = make_float2(p.x, __fmul_rn(p.x, p.x));
            const float yy = __fmul_rn(p.y, p.y);
#pragma unroll
            for (int r = 0; r < R; ++r) tile.yd[pos][r] = axis_sqdist(p.y, yy, cym2[r], cyy[r]);
            if (HAS_W) tile.aux[pos] = wi;
            if (HAS_IDX) tile.idx[pos] = (unsigned char)i;
        }
        kept += __popc(ballot);
    }
    return kept;
}

// Register prefetch of the NEXT tile of points (and weights): issued right after the current tile is staged, so the
// loads fly under the exponential loop.  Used by the small pixel tiles (R*C < 16), which have registers to spare and are
// what a rank of a sharded sweep runs: with about one task per resident warp the warps of an SM move through
// staging in step, and nobody else hides the round trip.  Indices are clamped like stage_points pads.
constexpr int PF = TILE_PTS / 32;
template <bool HAS_W>
__device__ __forceinline__ void fetch_points(const float2* __restrict__ pts, const float* __restrict__ w, int n0, int limit,
                                             float2 (&p)[PF], float (&wv)[PF]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int u = 0; u < PF; ++u) {
        const int n = min(n0 + 32 * u + lane, limit - 1);
        DGVCC_DEV_CHECK(n >= 0);
        p[u] = __ldg(&pts[n]);
        if (HAS_W) wv[u] = __ldg(&w[n]);
    }
}

// stage_points from prefetched registers.
template <int R>
__device__ __forceinline__ void stage_fetched(WarpTile<R>& tile, const float2 (&p)[PF], int padded, const float (&cym2)[R],
                                              const float (&cyy)[R]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int u = 0; u < PF; ++u) {
        const int i = 32 * u + lane;
        if (i < padded) {
            tile.xs[i] = make_float2(p[u].x, __fmul_rn(p[u].x, p[u].x));
            const float yy = __fmul_rn(p[u].y, p[u].y);
#pragma unroll
            for (int r = 0; r < R; ++r) tile.yd[i][r] = axis_sqdist(p[u].y, yy, cym2[r], cyy[r]);
        }
    }
}

// stage_points_if<R, true, false> from prefetched registers (weights in tile.aux, ordered compaction).
template <int R, typename Keep>
__device__ __forceinline__ int stage_fetched_if(WarpTile<R>& tile, const float2 (&p)[PF], const float (&wv)[PF], int cnt,
                                                const float (&cym2)[R], const float (&cyy)[R], Keep keep_fn) {
    const int lane = threadIdx.x & 31;
    int kept = 0;
#pragma unroll
    for (int u = 0; u < PF; ++u) {
        if (32 * u >= cnt) break;  // warp-uniform
        const int i = 32 * u + lane;
        const bool keep = i < cnt && keep_fn(p[u].x, p[u].y, wv[u]);
        const unsigned int ballot = __ballot_sync(FULL_MASK, keep);
        if (keep) {
            const int pos = kept + __popc(ballot & ((1u << lane) - 1u));
            DGVCC_DEV_CHECK(pos >= 0 && pos < TILE_PTS);
            tile.xs[pos] = make_float2(p[u].x, __fmul_rn(p[u].x, p[u].x));
            const float yy = __fmul_rn(p[u].y, p[u].y);
#pragma unroll
            for (int r = 0; r < R; ++r) tile.yd[pos][r] = axis_sqdist(p[u].y, yy, cym2[r], cyy[r]);
            tile.aux[pos] = wv[u];
        }
        kept += __popc(ballot);
    }
    return kept;
}

// Conservative lower bound of the reference's fp32 squared distance dis[n, pixel] over every pixel
// of a warp's tile, from the point's distance to the rectangle of the tile's cell centres.  The slack
// covers (i) the rounding of this bound itself and (ii) the error of the reference's cancelling
// expansion -2pc + p^2 + c^2 (<= 2^-21 (Mx + My), M = largest squared magnitude involved); 4x margin.
struct TileBox {
    float x0, x1, y0, y1;  // first / last cell centre of the tile per axis
    __device__ __forceinline__ float lower_bound(float x, float y) const {
        const float dx = fmaxf(fmaxf(x0 - x, x - x1), 0.f);
        const float dy = fmaxf(fmaxf(y0 - y, y - y1), 0.f);
        const float lb = fmaf(dx, dx, dy * dy);
        const float m = fmaxf(x * x, x1 * x1) + fmaxf(y * y, y1 * y1);
        return lb - fmaf(lb, 9.5367431640625e-07f /*2^-20*/, m * 1.9073486328125e-06f /*2^-19*/);
    }
};

template <int R>
__device__ __forceinline__ void load_yd(const WarpTile<R>& tile, int i, float (&yd)[R]) {
    if (R == 2) {
        const float2 v = *reinterpret_cast<const float2*>(&tile.yd[i][0]);
        yd[0] = v.x; yd[1] = v.y;
    } else {
#pragma unroll
        for (int q = 0; q < R / 4; ++q) {
            const float4 v = *reinterpret_cast<const float4*>(&tile.yd[i][4 * q]);
            yd[4 * q + 0] = v.x; yd[4 * q + 1] = v.y; yd[4 * q + 2] = v.z; yd[4 * q + 3] = v.w;
        }
    }
}

// The R y-distances of staged point i as R/2 packed pairs (rows 2q, 2q+1).
template <int R>
__device__ __forceinline__ void load_yd2(const WarpTile<R>& tile, int i, f2 (&yd)[R / 2]) {
    if (R == 2) {
        yd[0] = *reinterpret_cast<const f2*>(&tile.yd[i][0]);
    } else {
#pragma unroll
        for (int q = 0; q < R / 4; ++q) {
            const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(&tile.yd[i][4 * q]);
            yd[2 * q] = v.x; yd[2 * q + 1] = v.y;
        }
    }
}

// Per-thread constants of the pixel tile: R row centres, C column centres (as -2c and c*c).
// Pixel (r, c) of the thread is grid cell (row_base + r, col0 + 32 c); cells past the grid edge are
// clamped onto the last row / column (a finite duplicate that is computed but never stored).
template <int R, int C>
struct PixelTile {
    float cym2[R], cyy[R], cxm2[C], cxx[C];
    int col[C];       // clamped column index
    int row_base, hp, wp, col0;
    TileBox box;

    __device__ __forceinline__ void init(const TaskInfo& t, const Geom& g) {
        row_base = t.row_base; hp = g.hp; wp = g.wp; col0 = t.col0;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float cy = cell_centre(min(t.row_base + r, g.hp - 1), g);
            cym2[r] = -2.0f * cy;
            cyy[r] = __fmul_rn(cy, cy);
        }
#pragma unroll
        for (int c = 0; c < C; ++c) {
            col[c] = min(t.col0 + 32 * c, g.wp - 1);
            const float cx = cell_centre(col[c], g);
            cxm2[c] = -2.0f * cx;
            cxx[c] = __fmul_rn(cx, cx);
        }
        const int blk_col0 = t.col0 - (int)(threadIdx.x & 31);
        box.x0 = cell_centre(blk_col0, g);
        box.x1 = cell_centre(min(blk_col0 + 32 * C - 1, g.wp - 1), g);
        box.y0 = cell_centre(t.row_base, g);
        box.y1 = cell_centre(min(t.row_base + R - 1, g.hp - 1), g);
    }
    __device__ __forceinline__ int pix(int r, int c) const {
        DGVCC_DEV_CHECK(row_base >= 0 && col[c] >= 0 && col[c] < wp);
        return min(row_base + r, hp - 1) * wp + col[c];
    }
    __device__ __forceinline__ bool ok(int r, int c) const { return row_base + r < hp && col0 + 32 * c < wp; }
};

// Largest value of v[r][c] over the whole warp tile.
template <int R, int C>
__device__ __forceinline__ float tile_max(const float (&v)[R][C]) {
    float m = v[0][0];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) m = fmaxf(m, v[r][c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(FULL_MASK, m, o));
    return m;
}

// Exact-zero culling of the exponential sweeps (opt-in): exp(a - amax) is computed as one MUFU.EX2 with
// flush-to-zero, so it is exactly +0 whenever (a - amax) * log2(e) < -126.  With a <= -lb/s for every pixel
// of the tile and amax >= the tile's smallest amax, a point is skipped when that bound is below -128 --
// every term it would have contributed is an exact zero, and the results are bit-identical.
struct ExpCull {
    bool on;
    float k2_max;  // max over the tile of k2 = -amax * log2(e)
    float k1;      // -log2(e) / s
    TileBox box;
    __device__ __forceinline__ bool keep(float x, float y) const {
        if (!on) return true;
        return fmaf(box.lower_bound(x, y), k1, k2_max) >= -128.f;
    }
};

// ------------------------------------------------------------------------------------------ K0
// min_n dis[n, pixel] over ALL points of an image (bl.py:39), through a uniform grid over the points.
// The minimum is exact whatever the order of the points, so they may be visited by locality instead of by index:
//   bl_grid_build_kernel : one CTA per image sorts its points by grid cell (counting sort in shared memory; the order
//                          inside a cell is whatever the atomics give -- it cannot change a minimum);
//   bl_gridmin_kernel    : warp task = (image, pixel tile).  The warp visits the cells around its tile ring by ring
//                          (ring d = cells at Chebyshev cell distance d from the cells the tile's rectangle of pixel
//                          centres overlaps): every point of a ring is tested against the exact per-point lower bound
//                          of TileBox and, if it can still lower some pixel's minimum, swept over the tile.  Any point of
//                          a ring beyond d lies at least d cells away from the rectangle, so the walk stops as soon as
//                          the tile's largest current minimum is below that distance (minus the rounding slack of the
//                          reference's cancelling expansion).
// Measured on the config-3 batch: 70 us (13 build + 57 walk) against 83 us for the index-ordered per-chunk sweeps this
// replaces -- and there are no per-chunk minima to combine or, in the sharded path, to exchange: every rank finds the
// minima of the images it touches from the (replicated) points itself, which removes one of five exchange phases.
constexpr int GRID_MAX_CELLS = 4096;   // 4 cells per thread of bl_grid_build_kernel
constexpr int GRID_CELLS_PER_THREAD = GRID_MAX_CELLS / 1024;

struct GridGeom {
    float cell, inv_cell;   // cell side in image pixels (a power of two: cell indices are exact), its reciprocal
    int gx, gy;             // cells per row / column, gx * gy <= GRID_MAX_CELLS
    float slack_m;          // magnitude term of the ring bound's rounding slack (see TileBox::lower_bound)
};

__device__ __forceinline__ int grid_cell_1d(float v, float inv_cell, int n) {
    return min(max((int)floorf(v * inv_cell), 0), n - 1);   // points outside the grid fall into the border cells
}

__global__ void __launch_bounds__(1024)
bl_grid_build_kernel(const float2* __restrict__ pts_all, const int32_t* __restrict__ meta, int batch, GridGeom gg,
                     int img_first, int32_t* __restrict__ goff, float2* __restrict__ gsorted,
                     unsigned int* __restrict__ ztick, unsigned int* __restrict__ gtick, int tiles_img,
                     unsigned int* __restrict__ queue) {
    __shared__ int hist[GRID_MAX_CELLS];
    __shared__ int warp_tot[32];
    const int img = img_first + blockIdx.x, tid = threadIdx.x;
    // first kernel of every forward pass: the image's per-tile arrival counters (tile_last_arrival) start at zero
    // even if an earlier step was cut short
    for (int i = tid; i < tiles_img; i += 1024) {
        ztick[(size_t)img * tiles_img + i] = 0u;
        gtick[(size_t)img * tiles_img + i] = 0u;
    }
    if (blockIdx.x == 0 && tid < 6) queue[tid] = 0u;   // the work queues of the persistent sweeps
    const Meta mv = meta_view(meta, batch);
    const int pt0 = mv.pt_off[img], n = mv.pt_off[img + 1] - pt0;
    DGVCC_DEV_CHECK(img >= 0 && img < batch && pt0 >= 0 && n >= 0);
    DGVCC_DEV_CHECK(gg.gx >= 1 && gg.gy >= 1 && gg.gx * gg.gy <= GRID_MAX_CELLS);
    if (n == 0) return;
    const float2* pts = pts_all + pt0;
#pragma unroll
    for (int u = 0; u < GRID_CELLS_PER_THREAD; ++u) hist[tid + 1024 * u] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += 1024) {
        const float2 p = __ldg(pts + i);
        atomicAdd(&hist[grid_cell_1d(p.y, gg.inv_cell, gg.gy) * gg.gx + grid_cell_1d(p.x, gg.inv_cell, gg.gx)], 1);
    }
    __syncthreads();
    int cellc[GRID_CELLS_PER_THREAD], mine = 0;   // this thread's consecutive cells
#pragma unroll
    for (int u = 0; u < GRID_CELLS_PER_THREAD; ++u) {
        cellc[u] = hist[GRID_CELLS_PER_THREAD * tid + u];
        mine += cellc[u];
    }
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(FULL_MASK, incl, o);
        if ((tid & 31) >= o) incl += v;
    }
    if ((tid & 31) == 31) warp_tot[tid >> 5] = incl;
    __syncthreads();
    if (tid < 32) {
        const int w = warp_tot[tid];
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(FULL_MASK, wi, o);
            if (tid >= o) wi += v;
        }
        warp_tot[tid] = wi - w;
    }
    __syncthreads();
    int excl = warp_tot[tid >> 5] + incl - mine;
    int32_t* off = goff + (size_t)img * (GRID_MAX_CELLS + 1);
    __syncthreads();                       // every thread has read its cells' counts
#pragma unroll
    for (int u = 0; u < GRID_CELLS_PER_THREAD; ++u) {
        off[GRID_CELLS_PER_THREAD * tid + u] = excl;    // cells past gx * gy are empty: their offsets equal n
        hist[GRID_CELLS_PER_THREAD * tid + u] = excl;   // now the write cursor of the cell
        excl += cellc[u];
    }
    if (tid == 1023) off[GRID_MAX_CELLS] = n;
    __syncthreads();
    float2* out = gsorted + pt0;
    for (int i = tid; i < n; i += 1024) {
        const float2 p = __ldg(pts + i);
        const int slot = atomicAdd(&hist[grid_cell_1d(p.y, gg.inv_cell, gg.gy) * gg.gx + grid_cell_1d(p.x, gg.inv_cell, gg.gx)], 1);
        DGVCC_DEV_CHECK(slot >= 0 && slot < n);
        out[slot] = p;
    }
}

template <int R, int C>
__global__ void __launch_bounds__(CTA_THREADS)
bl_gridmin_kernel(const float2* __restrict__ gsorted, const int32_t* __restrict__ goff, const int32_t* __restrict__ meta,
                  int batch, Geom g, GridGeom gg, int img_first, float* __restrict__ min_img) {
    __shared__ WarpTile<R> tiles[WARPS_PER_CTA];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    TaskInfo t;
    t.task = g.task_first + blockIdx.x * WARPS_PER_CTA + warp;
    if (t.task >= g.tiles) return;
    t.img = img_first + blockIdx.y;
    const Meta mv = meta_view(meta, batch);
    const int pt0 = mv.pt_off[t.img], n = mv.pt_off[t.img + 1] - pt0;
    if (n == 0) return;
    t.col0 = (t.task % g.col_blocks) * 32 * C + lane;
    t.row_base = (t.task / g.col_blocks) * R;
    WarpTile<R>& tile = tiles[warp];
    PixelTile<R, C> px;
    px.init(t, g);
    const TileBox box = px.box;
    const int32_t* off = goff + (size_t)t.img * (GRID_MAX_CELLS + 1);
    const float2* sp = gsorted + pt0;
    const int cx0 = grid_cell_1d(box.x0, gg.inv_cell, gg.gx), cx1 = grid_cell_1d(box.x1, gg.inv_cell, gg.gx);
    const int cy0 = grid_cell_1d(box.y0, gg.inv_cell, gg.gy), cy1 = grid_cell_1d(box.y1, gg.inv_cell, gg.gy);
    float mind[R][C];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) mind[r][c] = __int_as_float(0x7f800000);
    int staged = 0;
    float bound = __int_as_float(0x7f800000);

    auto sweep_staged = [&]() {   // the staged points over the tile; refreshes the pruning bound
        __syncwarp();
#pragma unroll 2
        for (int i = 0; i < staged; ++i) {
            const float2 xs = tile.xs[i];
            float yd[R];
            load_yd<R>(tile, i, yd);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float xd = axis_sqdist(xs.x, xs.y, px.cxm2[c], px.cxx[c]);
#pragma unroll
                for (int r = 0; r < R; ++r) mind[r][c] = fminf(mind[r][c], __fadd_rn(yd[r], xd));
            }
        }
        staged = 0;
        bound = tile_max<R, C>(mind);
        __syncwarp();
    };
    // A ring is a handful of runs of consecutive cells (its top and bottom rows, two side cells per row in between);
    // the points of a run are consecutive in the sorted list.  Lane q looks up run q's point range -- all ranges of a
    // ring in ONE round trip to memory instead of one per run -- and the warp then walks the concatenation of the
    // ranges 32 points at a time (each lane finds its run by a 5-step search through the lanes' prefix sums).
    const int max_d = max(max(cx0, gg.gx - 1 - cx1), max(cy0, gg.gy - 1 - cy1));
    for (int d = 0; d <= max_d; ++d) {
        const int j_lo = max(cy0 - d, 0), j_hi = min(cy1 + d, gg.gy - 1);
        const int i_lo = max(cx0 - d, 0), i_hi = min(cx1 + d, gg.gx - 1);
        const bool top = d == 0 || cy0 - d >= 0, bottom = d > 0 && cy1 + d < gg.gy;        // full rows of the ring inside the grid
        const bool left = d > 0 && cx0 - d >= 0, right = d > 0 && cx1 + d < gg.gx;         // side columns inside the grid
        // run numbering: d == 0: one run per row; d > 0: [top row] [bottom row] then per middle row [left cell] [right cell]
        const int mid_lo = d == 0 ? 0 : max(cy0 - d + 1, 0), mid_hi = d == 0 ? -1 : min(cy1 + d - 1, gg.gy - 1);
        const int n_mid = max(mid_hi - mid_lo + 1, 0);
        const int n_runs = d == 0 ? (j_hi - j_lo + 1) : (2 + 2 * n_mid);
        for (int run0 = 0; run0 < n_runs; run0 += 32) {
            const int q = run0 + lane;
            int first = 0, count = 0;
            if (q < n_runs) {
                int c0 = -1, c1 = -1;   // cells [c0, c1] of the run, row-major
                if (d == 0) { c0 = (j_lo + q) * gg.gx + i_lo; c1 = (j_lo + q) * gg.gx + i_hi; }
                else if (q == 0) { if (top) { c0 = (cy0 - d) * gg.gx + i_lo; c1 = (cy0 - d) * gg.gx + i_hi; } }
                else if (q == 1) { if (bottom) { c0 = (cy1 + d) * gg.gx + i_lo; c1 = (cy1 + d) * gg.gx + i_hi; } }
                else {
                    const int jr = mid_lo + ((q - 2) >> 1);
                    if (((q - 2) & 1) == 0) { if (left) c0 = c1 = jr * gg.gx + cx0 - d; }
                    else if (right) c0 = c1 = jr * gg.gx + cx1 + d;
                }
                if (c0 >= 0) {
                    DGVCC_DEV_CHECK(c0 <= c1 && c1 < gg.gx * gg.gy && c1 < GRID_MAX_CELLS);
                    first = __ldg(off + c0);
                    count = __ldg(off + c1 + 1) - first;
                    DGVCC_DEV_CHECK(first >= 0 && count >= 0 && first + count <= n);
                }
            }
            int incl = count;   // prefix sums of the runs' lengths across the lanes
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(FULL_MASK, incl, o);
                if (lane >= o) incl += v;
            }
            const int total = __shfl_sync(FULL_MASK, incl, 31);
            const int excl = incl - count;
            // The candidates of a crowded ring are a long list (a cluster of 2000 heads is 63 batches of 32) and every
            // batch is a dependent L2 round trip: FOUR batches are looked up and loaded before the first is tested, so the
            // latency is paid once per 128 candidates (ncu, one rank of 8: the walk was 43 us of pure latency chain --
            // 9 % of the warp slots active -- with 15 us of grid build in front of it).
            constexpr int AHEAD = 4;
            for (int base = 0; base < total; base += 32 * AHEAD) {
                float2 pq[AHEAD];
#pragma unroll
                for (int u = 0; u < AHEAD; ++u) {
                    const int gi = base + 32 * u + lane;
                    // the run that holds concatenated index gi: the last lane whose exclusive prefix is <= gi
                    int lo = 0;
#pragma unroll
                    for (int step = 16; step > 0; step >>= 1) {
                        const int e = __shfl_sync(FULL_MASK, excl, min(lo + step, 31));
                        if (lo + step < 32 && e <= gi) lo += step;
                    }
                    const int r_first = __shfl_sync(FULL_MASK, first, lo), r_excl = __shfl_sync(FULL_MASK, excl, lo);
                    pq[u] = make_float2(0.f, 0.f);
                    DGVCC_DEV_CHECK(gi >= total || (gi >= r_excl && r_first + (gi - r_excl) < n));
                    if (gi < total) pq[u] = __ldg(sp + r_first + (gi - r_excl));
                }
#pragma unroll
                for (int u = 0; u < AHEAD; ++u) {
                    if (base + 32 * u >= total) break;   // warp-uniform
                    const int gi = base + 32 * u + lane;
                    const float2 p = pq[u];
                    const bool keep = gi < total && box.lower_bound(p.x, p.y) <= bound;
                    const unsigned int ballot = __ballot_sync(FULL_MASK, keep);
                    if (keep) {
                        const int pos = staged + __popc(ballot & ((1u << lane) - 1u));
                        DGVCC_DEV_CHECK(pos >= 0 && pos < TILE_PTS);
                        tile.xs[pos] = make_float2(p.x, __fmul_rn(p.x, p.x));
                        const float yy = __fmul_rn(p.y, p.y);
#pragma unroll
                        for (int r = 0; r < R; ++r) tile.yd[pos][r] = axis_sqdist(p.y, yy, px.cym2[r], px.cyy[r]);
                    }
                    staged += __popc(ballot);
                    if (staged > TILE_PTS - 32) sweep_staged();
                }
            }
        }
        sweep_staged();
        // every point not visited yet lies in a ring beyond d: at least d cells from the tile's rectangle
        const float far = (float)d * gg.cell, lb = far * far;
        if (bound <= lb - fmaf(lb, 9.5367431640625e-07f /*2^-20*/, gg.slack_m * 1.9073486328125e-06f /*2^-19*/)) break;
    }
    float* out = min_img + (size_t)t.img * g.hp * g.wp;
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c)
            if (px.ok(r, c)) out[px.pix(r, c)] = mind[r][c];
}

// The sweeps are persistent: a launch has at most as many CTAs as the GPU holds at once, and a warp (bl_z, bl_grad) or
// a CTA (bl_counts) that finishes a task takes the next one from a counter.  Work item w = (launch slot w / n, pixel
// tile or CTA of tiles w % n); the slots list the chunks longest first, so the queue is a longest-processing-time
// schedule: the sweep ends within one SHORT task of the moment the work runs out, instead of waiting for a last wave
// of full-length tasks.  queue[0] = items handed out beyond the first round, queue[1] = CTAs that left: the last one
// zeroes both for the next launch (bl_grid_build_kernel also zeroes them at the head of every forward pass).
__device__ __forceinline__ unsigned int queue_next_warp(unsigned int* queue, unsigned int first_round) {
    unsigned int w = 0u;
    if ((threadIdx.x & 31) == 0) w = first_round + atomicAdd(queue, 1u);
    return __shfl_sync(FULL_MASK, w, 0);
}
__device__ __forceinline__ void queue_leave(unsigned int* queue) {  // every thread of the CTA, after its last item
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(queue + 1, 1u) == gridDim.x - 1u) {
        queue[0] = 0u;
        queue[1] = 0u;
    }
}

// The chunks of one image sweep the same pixel tile in separate warp tasks; whichever task arrives LAST at the tile's
// counter combines the per-chunk partials (in chunk order, whoever does it: the sum does not depend on the arrival
// order) -- the classic last-block reduction, per pixel tile.  Saves a reduction kernel and a second pass over the
// partials; the counters are zeroed by bl_grid_build_kernel at the head of every forward pass and by the last arriver.
__device__ __forceinline__ bool tile_last_arrival(unsigned int* counter, int n_chunks) {
    __threadfence();   // this task's partials before its arrival
    __syncwarp();
    unsigned int old = 0u;
    if ((threadIdx.x & 31) == 0) old = atomicAdd(counter, 1u);
    old = __shfl_sync(FULL_MASK, old, 0);
    DGVCC_DEV_CHECK(n_chunks >= 1 && old < (unsigned)n_chunks);   // a counter left over from a step that was cut short
    const bool last = old == (unsigned)n_chunks - 1u;
    if (last) {
        if ((threadIdx.x & 31) == 0) *counter = 0u;
        __threadfence();   // the other tasks' partials after their arrivals
    }
    return last;
}

// What the last arrival does, kept out of line so that the sweeps' register allocation is that of their inner loops:
// the warp re-derives its pixels from (row_base, col0) and walks the chunks with all of a chunk's R*C loads in flight.
template <int R, int C>
__device__ __noinline__ void finish_z_tile(const float* __restrict__ zc, int n_chunks, size_t M, int row_base, int col0, int hp,
                                           int wp, const float* __restrict__ ebg_img, float* __restrict__ rz_img,
                                           float* __restrict__ pbg_img) {
    // 1 / (sum of the chunk shares in chunk order + background term last), the reference's row order (bl.py:44)
    int pix[R][C];
    float z[R][C];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            pix[r][c] = min(row_base + r, hp - 1) * wp + min(col0 + 32 * c, wp - 1);  // outside the grid: the clamped twin
            z[r][c] = 0.f;
        }
#pragma unroll 4
    for (int ch = 0; ch < n_chunks; ++ch, zc += M) {
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int c = 0; c < C; ++c) z[r][c] += __ldcg(zc + pix[r][c]);
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            if (row_base + r >= hp || col0 + 32 * c >= wp) continue;
            const float ebg = __ldcg(ebg_img + pix[r][c]);
            const float rz = 1.0f / (z[r][c] + ebg);
            rz_img[pix[r][c]] = rz;
            pbg_img[pix[r][c]] = ebg * rz;
        }
}

// Gradient of a multi-chunk image's pixel tile: chunk sums added in chunk order, per-pixel factors applied.
template <int R, int C>
__device__ __noinline__ void finish_grad_tile(const float* __restrict__ gc, int n_chunks, size_t M, int row_base, int col0,
                                              int hp, int wp, float gscale, float w_bg, const float* __restrict__ rz_img,
                                              const float* __restrict__ pbg_img, float* __restrict__ gout_img) {
    int pix[R][C];
    float a[R][C];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            pix[r][c] = min(row_base + r, hp - 1) * wp + min(col0 + 32 * c, wp - 1);
            a[r][c] = 0.f;
        }
#pragma unroll 4
    for (int ch = 0; ch < n_chunks; ++ch, gc += M) {
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int c = 0; c < C; ++c) a[r][c] += __ldcg(gc + pix[r][c]);
    }
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            if (row_base + r >= hp || col0 + 32 * c >= wp) continue;
            gout_img[pix[r][c]] = gscale * fmaf(a[r][c], rz_img[pix[r][c]], w_bg * pbg_img[pix[r][c]]);
        }
}

// ------------------------------------------------------------------------------------------ K1
// Softmax max (incl. the background row, bl.py:39-43) and this chunk's share of the denominator.
template <int R, int C, bool POW2>
__device__ __forceinline__ bool bl_z_body(const float2* __restrict__ pts_all, const int32_t* __restrict__ meta,
            const float* __restrict__ st_sizes, int batch, const Geom& g, const Scale& k, float bg_ratio, int use_bg,
            int exact_cull, float* __restrict__ zpart,
            float* __restrict__ amax_out, float* __restrict__ ebg_out, unsigned int* __restrict__ ticket, const Shard& sh,
            const float* __restrict__ min_img, const Xchg& x, float* __restrict__ rz_out, float* __restrict__ pbg_out,
            unsigned int* __restrict__ tile_tick, int finish, int slot, int task) {
    __shared__ WarpTile<R> tiles[WARPS_PER_CTA];
    TaskInfo t;
    if (!decode_task<R, C>(meta, batch, g, t, slot, task)) return false;
    WarpTile<R>& tile = tiles[threadIdx.x >> 5];
    const size_t M = (size_t)g.hp * g.wp;
    PixelTile<R, C> px;
    px.init(t, g);
    float* zout = zpart + (size_t)t.chunk * M;
    float* amax_img = amax_out + (size_t)t.img * M;
    float* ebg_img = ebg_out + (size_t)t.img * M;

    if (t.n_img_pts == 0) {  // bl.py:63-65: the only row is "sum of density": posterior == 1
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int c = 0; c < C; ++c)
                if (px.ok(r, c)) {
                    const int p = px.pix(r, c);
                    zout[p] = 0.f; amax_img[p] = 0.f; ebg_img[p] = 1.f;
                    if (finish) { rz_out[(size_t)t.img * M + p] = 1.f; pbg_out[(size_t)t.img * M + p] = 1.f; }  // 1 / (0 + 1)
                }
        return false;
    }
    const float2* pts = pts_all + t.pt_base;
    constexpr bool PREFETCH = R * C < 16;
    float2 pf[PF];
    float pw[PF];
    if (PREFETCH && !exact_cull && t.p_cnt > 0) fetch_points<false>(pts, nullptr, 0, t.p_cnt, pf, pw);  // under the prologue

    float neg_amax[R][C];  // first holds min dis, then k2 = -amax * log2(e)
    {  // bl_gridmin_kernel has been over the image
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int c = 0; c < C; ++c) neg_amax[r][c] = min_img[(size_t)t.img * M + px.pix(r, c)];
    }

    float ebg_arg[R][C], amax_v[R][C];  // (a_bg - amax) * log2(e); amax itself (stored for the later sweeps)
    const float dbg = __fmul_rn(st_sizes[t.img], bg_ratio);
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float mind = neg_amax[r][c];
            float amax = neg_div<POW2>(mind, k);
            float a_bg = 0.f;
            if (use_bg) {
                const float root = __fsqrt_rn(fmaxf(mind, 0.0f));
                const float diff = __fadd_rn(dbg, -root);
                a_bg = neg_div<POW2>(__fmul_rn(diff, diff), k);
                amax = fmaxf(amax, a_bg);
            }
            amax_v[r][c] = amax;
            neg_amax[r][c] = __fmul_rn(-amax, LOG2E);                    // k2 of pair_exp
            ebg_arg[r][c] = __fmaf_rn(a_bg, LOG2E, neg_amax[r][c]);     // same form as the point rows
        }

    // denominator share, accumulated in point order like torch's dim-0 softmax
    float z[R][C];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) z[r][c] = 0.f;
    const ExpCull cull{exact_cull != 0, tile_max<R, C>(neg_amax), k.k1, px.box};
    const Scale2 k2s(k);
    f2 zp[R / 2][C], k2p[R / 2][C];
#pragma unroll
    for (int q = 0; q < R / 2; ++q)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            zp[q][c] = pack2(0.f, 0.f);
            k2p[q][c] = pack2(neg_amax[2 * q][c], neg_amax[2 * q + 1][c]);
        }
    for (int n0 = 0; n0 < t.p_cnt; n0 += TILE_PTS) {
        int cnt = min(TILE_PTS, t.p_cnt - n0);
        __syncwarp();
        if (exact_cull)
            cnt = stage_points_if<R, false, false>(tile, pts, nullptr, n0, cnt, px.cym2, px.cyy,
                                                   [&](float x, float y, float) { return cull.keep(x, y); });
        else if (PREFETCH) {
            stage_fetched<R>(tile, pf, cnt, px.cym2, px.cyy);
            if (n0 + TILE_PTS < t.p_cnt) fetch_points<false>(pts, nullptr, n0 + TILE_PTS, t.p_cnt, pf, pw);
        } else
            stage_points<R>(tile, pts, n0, t.p_cnt, cnt, px.cym2, px.cyy);
        __syncwarp();
#pragma unroll 2
        for (int i = 0; i < cnt; ++i) {
            const float2 xs = tile.xs[i];
            f2 yd[R / 2];
            load_yd2<R>(tile, i, yd);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float xd = axis_sqdist(xs.x, xs.y, px.cxm2[c], px.cxx[c]);
                const f2 xd2 = pack2(xd, xd);
#pragma unroll
                for (int q = 0; q < R / 2; ++q) zp[q][c] = add2(zp[q][c], pair_exp2<POW2>(add2(yd[q], xd2), k2p[q][c], k2s));
            }
        }
    }
#pragma unroll
    for (int q = 0; q < R / 2; ++q)
#pragma unroll
        for (int c = 0; c < C; ++c) unpack2(zp[q][c], z[2 * q][c], z[2 * q + 1][c]);
    const bool first = t.chunk == max(t.first_chunk, sh.chunk_lo);  // the image's first chunk ON THIS RANK
    const unsigned int dst = x.peers ? x.mask[t.chunk] : 0u;
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            if (!px.ok(r, c)) continue;
            const int p = px.pix(r, c);
            zout[p] = z[r][c];
            if (first) {
                amax_img[p] = amax_v[r][c];
                ebg_img[p] = use_bg ? ex2_ftz(ebg_arg[r][c]) : 0.f;
            }
        }
    // the task that arrives last at the pixel tile turns the chunk shares into 1 / denominator (the image's first chunk
    // stored ebg before it arrived); out of line, see finish_z_tile
    if (finish && (t.n_chunks == 1 || tile_last_arrival(tile_tick + (size_t)t.img * g.tiles_img + t.task, t.n_chunks)))
        finish_z_tile<R, C>(zpart + (size_t)t.first_chunk * M, t.n_chunks, M, t.row_base, t.col0, g.hp, g.wp, ebg_img,
                            rz_out + (size_t)t.img * M, pbg_out + (size_t)t.img * M);
    for (unsigned int m = dst; m; m &= m - 1u) {  // the same tile into the workspaces of the image's other ranks
        float* rp = xchg_ptr(x, __ffs(m) - 1, x.region_off) + (size_t)t.chunk * M;
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int c = 0; c < C; ++c)
                if (px.ok(r, c)) rp[px.pix(r, c)] = z[r][c];
    }
    return dst != 0u;
}

template <int R, int C, bool POW2>
__global__ void __launch_bounds__(CTA_THREADS, 4)   // 16 warps per SM: <= 128 registers
bl_z_kernel(const float2* __restrict__ pts_all, const int32_t* __restrict__ meta,
            const float* __restrict__ st_sizes, int batch, Geom g, Scale k, float bg_ratio, int use_bg,
            int exact_cull, float* __restrict__ zpart,
            float* __restrict__ amax_out, float* __restrict__ ebg_out, unsigned int* __restrict__ ticket, Shard sh,
            const float* __restrict__ min_img, Xchg x, float* __restrict__ rz_out, float* __restrict__ pbg_out,
            unsigned int* __restrict__ tile_tick, int finish, int n_slots, unsigned int* __restrict__ queue) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *ticket = 0u;  // bl_select_kernel's arrival counter
    const int n_tiles = g.tiles - g.task_first;
    const unsigned int total = (unsigned)n_slots * (unsigned)n_tiles, first_round = gridDim.x * WARPS_PER_CTA;
    bool stored = false;
    for (unsigned int w = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5); w < total; w = queue_next_warp(queue, first_round)) {
        stored |= bl_z_body<R, C, POW2>(pts_all, meta, st_sizes, batch, g, k, bg_ratio, use_bg, exact_cull, zpart, amax_out,
                                        ebg_out, ticket, sh, min_img, x, rz_out, pbg_out, tile_tick, finish,
                                        (int)(w / n_tiles), g.task_first + (int)(w % n_tiles));
        __syncwarp();  // the warp's shared-memory tile is reused by its next task
    }
    queue_leave(queue);
    xchg_signal(x, stored);
}

// 1 / (sum of the chunk shares in chunk order + background term last), the reference's row order.
__device__ __forceinline__ float softmax_rz(const float* __restrict__ zpart, size_t M, int first_chunk, int n_chunks,
                                            int pix, float ebg) {
    float z = 0.f;
#pragma unroll 1
    for (int c = 0; c < n_chunks; ++c) z += zpart[(size_t)(first_chunk + c) * M + pix];
    return 1.0f / (z + ebg);
}

// ------------------------------------------------------------------------------------------ K2
// One partial count: into this GPU's cpart, or (row-band sharding) into the count-share table of every rank.
__device__ __forceinline__ void put_count(float* __restrict__ cpart, bool shared, const Xchg& x, size_t idx, float v) {
    if (!shared) {
        cpart[idx] = v;
    } else {
#pragma unroll 1
        for (int q = 0; q < x.world; ++q) xchg_ptr(x, q, x.region_off)[idx] = v;
    }
}

template <int R, int C, bool POW2>
__global__ void __launch_bounds__(CTA_THREADS, 5)   // 5 CTAs per SM (what the 39 KB of shared memory allow): <= 102 registers
bl_counts_kernel(const float2* __restrict__ pts_all, const int32_t* __restrict__ meta,
                 const float* __restrict__ density, int batch, Geom g, Scale k, int use_bg, int exact_cull,
                 const float* __restrict__ amax_in, const float* __restrict__ rz_in, const float* __restrict__ pbg_in,
                 int64_t total_rows, float* __restrict__ cpart, int share_row0, Xchg x, int n_slots,
                 unsigned int* __restrict__ queue) {
    xchg_wait(x);  // row-band sharding: the density rows of the band, delivered by the images' owners
    // The four warps of a CTA sweep the same point chunk over four pixel tiles; their per-point partial counts
    // meet in shared memory and leave the CTA as ONE partial row (a quarter of the cpart traffic, and a quarter
    // of what bl_reduce_counts_kernel has to read).  Warps past the last pixel tile contribute zeros.
    // share_row0 >= 0 (row-band sharding): the partial row is row share_row0 + blockIdx.x of the count-share table and
    // goes, as it is produced, into the table of EVERY rank (plain stores over NVLink); the last CTA raises the flag.
    __shared__ WarpTile<R> tiles[WARPS_PER_CTA];
    __shared__ float cta_acc[WARPS_PER_CTA][COUNT_SPAN];
    __shared__ float cta_bg[WARPS_PER_CTA];
    __shared__ unsigned int next_item;
    const int warp = threadIdx.x >> 5;
    WarpTile<R>& tile = tiles[warp];
    const int lane = threadIdx.x & 31;
    const size_t M = (size_t)g.hp * g.wp;
    // persistent CTAs: item = (launch slot, CTA of four pixel tiles), see queue_next_warp
    const int n_ctas = ceil_div(g.tiles - g.task_first, WARPS_PER_CTA);
    const unsigned int total_items = (unsigned)n_slots * (unsigned)n_ctas;
    for (unsigned int item = blockIdx.x; item < total_items;) {
    const int cta_x = (int)(item % n_ctas);
    TaskInfo t;
    const bool live = decode_task<R, C>(meta, batch, g, t, (int)(item / n_ctas), g.task_first + cta_x * WARPS_PER_CTA + warp);
    const size_t img_base = (size_t)t.img * M;
    PixelTile<R, C> px;
    px.init(t, g);
    const size_t part0 = (size_t)(max(share_row0, 0) + cta_x) * total_rows + t.row0;
    DGVCC_DEV_CHECK(cta_x >= 0 && t.row0 + t.n_rows <= total_rows && t.p_start + t.p_cnt <= t.n_rows);
    const bool bg_row = t.chunk == t.first_chunk && (use_bg || t.n_img_pts == 0);  // the image's first chunk anywhere

    // per-pixel weights D[m]/Z[m]; pixels outside the grid get weight 0
    float neg_amax[R][C], wd[R][C], bg_part = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int p = px.pix(r, c);
            const size_t m = img_base + p;
            const bool ok = live && px.ok(r, c);
            const float d = ok ? density[m] : 0.f;
            const float rz = rz_in[m], pbg = pbg_in[m];  // finished by bl_z_kernel's last arrival (or bl_finish_z_kernel)
            neg_amax[r][c] = __fmul_rn(-amax_in[m], LOG2E);
            // a pixel outside the grid -- or, for the idle warps of a band's last CTA, outside the band, where this rank
            // holds no denominators at all -- must not leak a NaN through 0 * inf
            wd[r][c] = ok ? d * rz : 0.f;
            if (ok) bg_part = fmaf(d, pbg, bg_part);
        }
    if (bg_row) {  // background row / sum-of-density row of an empty image
        bg_part = warp_sum(bg_part);
        if (lane == 0) cta_bg[warp] = bg_part;
    }
    __syncthreads();
    if (bg_row && threadIdx.x == 0)
        put_count(cpart, share_row0 >= 0, x, part0 + t.n_rows - 1, ((cta_bg[0] + cta_bg[1]) + cta_bg[2]) + cta_bg[3]);

    const float2* pts = pts_all + t.pt_base;
    const ExpCull cull{exact_cull != 0, tile_max<R, C>(neg_amax), k.k1, px.box};
    const Scale2 k2s(k);
    f2 k2p[R / 2][C], wdp[R / 2][C];
#pragma unroll
    for (int q = 0; q < R / 2; ++q)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            k2p[q][c] = pack2(neg_amax[2 * q][c], neg_amax[2 * q + 1][c]);
            wdp[q][c] = pack2(wd[2 * q][c], wd[2 * q + 1][c]);
        }
    constexpr bool PREFETCH = R * C < 16;
    float2 pf[PF];
    float pw[PF];
    if (PREFETCH && live && !exact_cull && t.p_cnt > 0) fetch_points<false>(pts, nullptr, 0, t.p_cnt, pf, pw);
    for (int span0 = 0; span0 < t.p_cnt; span0 += COUNT_SPAN) {
        const int span_cnt = min(COUNT_SPAN, t.p_cnt - span0);
        if (!live)
            for (int i = lane; i < span_cnt; i += 32) cta_acc[warp][i] = 0.f;
        for (int n0 = span0; live && n0 < span0 + span_cnt; n0 += TILE_PTS) {
            const int cnt = min(TILE_PTS, t.p_cnt - n0);
            float* acc_w = &cta_acc[warp][n0 - span0];
            int kept = cnt;
            __syncwarp();
            if (exact_cull) {
                for (int i = lane; i < cnt; i += 32) acc_w[i] = 0.f;  // culled points: partial count exactly 0
                kept = stage_points_if<R, false, true>(tile, pts, nullptr, n0, cnt, px.cym2, px.cyy,
                                                       [&](float x, float y, float) { return cull.keep(x, y); });
                __syncwarp();
                // pad the compacted list to a multiple of 8 with copies of its last point (results discarded)
                for (int i = kept + lane; i < ((kept + 7) & ~7); i += 32) {
                    tile.xs[i] = tile.xs[kept - 1];
#pragma unroll
                    for (int r = 0; r < R; ++r) tile.yd[i][r] = tile.yd[kept - 1][r];
                }
            } else if (PREFETCH) {
                stage_fetched<R>(tile, pf, (cnt + 7) & ~7, px.cym2, px.cyy);
                if (n0 + TILE_PTS < t.p_cnt) fetch_points<false>(pts, nullptr, n0 + TILE_PTS, t.p_cnt, pf, pw);
            } else {
                stage_points<R>(tile, pts, n0, t.p_cnt, (cnt + 7) & ~7, px.cym2, px.cyy);
            }
            const int padded = (kept + 7) & ~7;
            __syncwarp();
#pragma unroll 1
            for (int i0 = 0; i0 < padded; i0 += 8) {
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float2 xs = tile.xs[i0 + u];
                    f2 yd[R / 2];
                    load_yd2<R>(tile, i0 + u, yd);
                    f2 s2 = pack2(0.f, 0.f);  // even / odd rows accumulate side by side
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const float xd = axis_sqdist(xs.x, xs.y, px.cxm2[c], px.cxx[c]);
                        const f2 xd2 = pack2(xd, xd);
#pragma unroll
                        for (int q = 0; q < R / 2; ++q)
                            s2 = fma2(pair_exp2<POW2>(add2(yd[q], xd2), k2p[q][c], k2s), wdp[q][c], s2);
                    }
                    float s_even, s_odd;
                    unpack2(s2, s_even, s_odd);
                    v[u] = s_even + s_odd;
                }
                // transpose-reduce: 8 per-lane partials -> lane quad q holds the warp total of point i0+q
#pragma unroll
                for (int h = 4, bit = 16; h >= 1; h >>= 1, bit >>= 1) {
                    const bool up = (lane & bit) != 0;
#pragma unroll
                    for (int u = 0; u < h; ++u) {
                        const float send = up ? v[u] : v[u + h];
                        const float keep = up ? v[u + h] : v[u];
                        v[u] = keep + __shfl_xor_sync(FULL_MASK, send, bit);
                    }
                }
                v[0] += __shfl_xor_sync(FULL_MASK, v[0], 2);
                v[0] += __shfl_xor_sync(FULL_MASK, v[0], 1);
                if ((lane & 3) == 0) {
                    const int q = i0 + (lane >> 2);
                    DGVCC_DEV_CHECK(n0 - span0 >= 0 && n0 - span0 + cnt <= COUNT_SPAN && q < TILE_PTS);
                    DGVCC_DEV_CHECK(!exact_cull || q >= kept || (int)tile.idx[q] < cnt);
                    if (!exact_cull) { if (q < cnt) acc_w[q] = v[0]; }
                    else if (q < kept) acc_w[tile.idx[q]] = v[0];
                }
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < span_cnt; i += CTA_THREADS)
            put_count(cpart, share_row0 >= 0, x, part0 + t.p_start + span0 + i,
                      ((cta_acc[0][i] + cta_acc[1][i]) + cta_acc[2][i]) + cta_acc[3][i]);
        __syncthreads();
    }
    if (threadIdx.x == 0) next_item = gridDim.x + atomicAdd(queue, 1u);
    __syncthreads();
    item = next_item;
    __syncthreads();   // everybody has read next_item before thread 0 can overwrite it
    }
    queue_leave(queue);
    xchg_signal(x, share_row0 >= 0);
}

// ------------------------------------------------------------------------------------------ K3
constexpr int SELECT_THREADS = 1024;
constexpr int SELECT_REGS = 12;   // residuals a thread keeps in registers across the radix passes (12 288 rows per image)

__device__ __forceinline__ float block_sum_ordered(float v, float* scratch) {
    // deterministic: warp butterfly, then warp partials added in warp order by thread 0
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    float total = 0.f;
    if (threadIdx.x == 0)
        for (int w = 0; w < SELECT_THREADS / 32; ++w) total += scratch[w];
    return total;  // valid on thread 0
}

// Expected counts: fixed-order sum of the per-tile partials (one thread per posterior row, coalesced
// across rows), and the residual |t - c|  (bl.py:73-75).
__device__ __forceinline__ bool bl_reduce_counts_body(const float* __restrict__ cpart, int tiles, int64_t total_rows,
                        const int32_t* __restrict__ meta, const float* __restrict__ targets, int batch,
                        float* __restrict__ counts, float* __restrict__ residual, const Shard& sh, const Xchg& x,
                        int64_t row_first);

__global__ void __launch_bounds__(256)
bl_reduce_counts_kernel(const float* __restrict__ cpart, int tiles, int64_t total_rows,
                        const int32_t* __restrict__ meta, const float* __restrict__ targets, int batch,
                        float* __restrict__ counts, float* __restrict__ residual, Shard sh, Xchg x, int64_t row_first) {
    const bool stored = bl_reduce_counts_body(cpart, tiles, total_rows, meta, targets, batch, counts, residual, sh, x, row_first);
    xchg_signal(x, stored);
}

__device__ __forceinline__ bool bl_reduce_counts_body(const float* __restrict__ cpart, int tiles, int64_t total_rows,
                        const int32_t* __restrict__ meta, const float* __restrict__ targets, int batch,
                        float* __restrict__ counts, float* __restrict__ residual, const Shard& sh, const Xchg& x,
                        int64_t row_first) {
    const int64_t j = row_first + (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= total_rows) return false;
    const Meta mv = meta_view(meta, batch);
    int lo = 0, hi = batch;  // image of row j: row_off[lo] <= j < row_off[lo+1]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (mv.row_off[mid] <= j) lo = mid; else hi = mid;
    }
    const int local = (int)(j - mv.row_off[lo]);
    const int n_pts = mv.pt_off[lo + 1] - mv.pt_off[lo];
    DGVCC_DEV_CHECK(j >= 0 && local >= 0 && j < mv.row_off[lo + 1] && local <= n_pts && tiles >= 1);
    if (sh.on) {  // only rows whose partials this rank computed: its own points; the last row with the image's first chunk
        const int gp = mv.pt_off[lo] + local;
        const bool mine = local < n_pts ? (gp >= sh.pt_lo && gp < sh.pt_hi)
                                        : (mv.icb[lo] >= sh.chunk_lo && mv.icb[lo] < sh.chunk_hi);
        if (!mine) return false;
    }
    const float* p = cpart + j;
    float c = 0.f;
#pragma unroll 8
    for (int tl = 0; tl < tiles; ++tl) c += p[(size_t)tl * total_rows];
    const float tgt = (local < n_pts) ? targets[mv.pt_off[lo] + local] : 0.f;
    const float res = fabsf(__fadd_rn(tgt, -c));
    counts[j] = c;
    residual[j] = res;
    if (x.peers) {  // the image's other ranks need every row for the top-k cut (bl.py:77)
        const unsigned int dst = x.mask[lo];
        xchg_store(x, dst, x.region_off, (size_t)j, c);
        xchg_store(x, dst, x.region_off2, (size_t)j, res);
        return dst != 0u;
    }
    return false;
}

__global__ void __launch_bounds__(SELECT_THREADS)
bl_select_kernel(const int32_t* __restrict__ meta, const float* __restrict__ targets, int batch,
                 float inv_batch, const float* __restrict__ counts, const float* __restrict__ residual,
                 float* __restrict__ wsel, float* __restrict__ loss_img, float* __restrict__ loss_out,
                 unsigned int* __restrict__ ticket, int img_first, int finish, Shard sh, Xchg x, int n_img) {
    xchg_wait(x);  // sharded: the counts / residuals of the rows other ranks computed
    if ((int)blockIdx.x >= n_img) {  // a rank that touches no image still takes part in the exchange
        xchg_signal(x);
        return;
    }
    __shared__ unsigned int hist[256];
    __shared__ unsigned int sh_prefix, sh_rank, sh_equal;
    __shared__ unsigned int warp_cnt[SELECT_THREADS / 32];
    __shared__ float scratch[SELECT_THREADS / 32];

    const int img = img_first + blockIdx.x, tid = threadIdx.x;
    const Meta mv = meta_view(meta, batch);
    const int pt0 = mv.pt_off[img], n_pts = mv.pt_off[img + 1] - pt0;
    const int row0 = mv.row_off[img], n_rows = mv.row_off[img + 1] - row0;
    const int n_cand = n_rows - 1;  // res[:-1]; the last row is always kept (bl.py:77-78)
    const int n_keep = mv.keep[img];
    DGVCC_DEV_CHECK(img >= 0 && img < batch && n_rows >= 1 && n_pts >= 0 && n_pts <= n_rows && n_keep <= max(n_cand, 0));

    // k-th smallest residual among the candidates: MSB-first radix select on the float bits
    unsigned int thr = 0xffffffffu;  // keep everything
    unsigned int take_equal = 0xffffffffu, n_equal = 0;
    if (n_keep <= 0) {
        thr = 0u; take_equal = 0u;  // keep nothing (residuals are >= +0, none is < 0)
    } else if (n_keep < n_cand) {
        if (tid == 0) { sh_prefix = 0u; sh_rank = (unsigned)n_keep; }
        // the four radix passes read the residuals from registers: up to SELECT_REGS per thread are loaded ONCE, all
        // loads in flight together (re-reading them from L2 in every pass was a chain of 4 x 12 load latencies for a
        // 12 000-row image); longer images read the tail from memory in every pass
        unsigned int held[SELECT_REGS];
#pragma unroll
        for (int u = 0; u < SELECT_REGS; ++u) {
            const int j = tid + u * SELECT_THREADS;
            held[u] = j < n_cand ? __float_as_uint(residual[row0 + j]) : 0u;
        }
        unsigned int mask = 0u;
        for (int shift = 24; shift >= 0; shift -= 8) {
            for (int b = tid; b < 256; b += SELECT_THREADS) hist[b] = 0u;
            __syncthreads();
            const unsigned int prefix = sh_prefix;
#pragma unroll
            for (int u = 0; u < SELECT_REGS; ++u)
                if (tid + u * SELECT_THREADS < n_cand && (held[u] & mask) == prefix) atomicAdd(&hist[(held[u] >> shift) & 255u], 1u);
            for (int j = tid + SELECT_REGS * SELECT_THREADS; j < n_cand; j += SELECT_THREADS) {
                const unsigned int bits = __float_as_uint(residual[row0 + j]);
                if ((bits & mask) == prefix) atomicAdd(&hist[(bits >> shift) & 255u], 1u);
            }
            __syncthreads();
            if (tid < 32) {  // first bin whose running count reaches the rank: 8 bins per lane + a warp scan
                const unsigned int rank = sh_rank;
                unsigned int h[8], mine = 0u;
#pragma unroll
                for (int u = 0; u < 8; ++u) { h[u] = hist[8 * tid + u]; mine += h[u]; }
                unsigned int incl = mine;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned int up = __shfl_up_sync(FULL_MASK, incl, o);
                    if (tid >= o) incl += up;
                }
                unsigned int cum = incl - mine;
                if (cum < rank && rank <= incl) {  // exactly one lane (the matching elements number >= rank)
                    int u = 0;
                    for (; u < 7; ++u) {
                        if (cum + h[u] >= rank) break;
                        cum += h[u];
                    }
                    sh_rank = rank - cum;
                    sh_prefix = prefix | ((unsigned)(8 * tid + u) << shift);
                    sh_equal = h[u];
                }
            }
            mask |= 255u << shift;
            __syncthreads();
        }
        thr = sh_prefix; take_equal = sh_rank; n_equal = sh_equal;
    }
    const bool ordered_ties = (n_keep > 0 && n_keep < n_cand && take_equal < n_equal);

    // selection, signed weights for backward, per-image loss
    float lsum = 0.f;
    unsigned int ties_seen = 0u;
    for (int base = 0; base < n_rows; base += SELECT_THREADS) {
        const int j = base + tid;
        const bool live = j < n_rows;
        float res = 0.f, c = 0.f, tgt = 0.f;
        unsigned int bits = 0u;
        if (live) {
            res = residual[row0 + j];
            c = counts[row0 + j];
            tgt = (j < n_pts) ? targets[pt0 + j] : 0.f;
            bits = __float_as_uint(res);
        }
        const bool cand = live && j < n_cand;
        bool tie_ok = true;
        if (ordered_ties) {  // equal residuals straddle the cut: keep the first `take_equal` in index order
            const bool is_tie = cand && bits == thr;
            const unsigned int ballot = __ballot_sync(FULL_MASK, is_tie);
            if ((tid & 31) == 0) warp_cnt[tid >> 5] = __popc(ballot);
            __syncthreads();
            unsigned int before = ties_seen, total = 0u;
            for (int w = 0; w < SELECT_THREADS / 32; ++w) {
                if (w < (tid >> 5)) before += warp_cnt[w];
                total += warp_cnt[w];
            }
            before += __popc(ballot & ((1u << (tid & 31)) - 1u));
            tie_ok = before < take_equal;
            ties_seen += total;
            __syncthreads();
        }
        bool sel = false;
        if (live) {
            if (j == n_rows - 1) sel = true;
            else sel = (bits < thr) || (bits == thr && take_equal > 0u && tie_ok);
            const float x = __fadd_rn(tgt, -c);  // d|x|/dc = -sign(x)
            const float w = sel ? (x > 0.f ? -1.f : (x < 0.f ? 1.f : 0.f)) : 0.f;
            wsel[row0 + j] = w;
            if (sel) lsum += res;
        }
    }
    const float l_img = block_sum_ordered(lsum, scratch);

    // last CTA to finish adds the per-image losses in image order (deterministic), bl.py:79
    if (tid == 0 && !finish) {  // sharded: bl_loss_finish_kernel adds the images' losses once every rank's have arrived
        loss_img[img] = l_img;
        const int first_chunk = mv.icb[img];
        if (x.peers && first_chunk >= sh.chunk_lo && first_chunk < sh.chunk_hi)  // from the rank with the image's first chunk
            xchg_store(x, ((1u << x.world) - 1u) & ~(1u << x.rank), x.region_off, (size_t)img, l_img);
    }
    if (!finish) xchg_signal(x);
    if (tid == 0 && finish) {
        loss_img[img] = l_img;
        __threadfence();
        const unsigned int done = atomicAdd(ticket, 1u);
        if (done == (unsigned)batch - 1u) {
            __threadfence();
            float total = 0.f;
            const volatile float* li = loss_img;
            for (int i = 0; i < batch; ++i) total += li[i];
            loss_out[0] = total * inv_batch;
            *ticket = 0u;
        }
    }
}

// ------------------------------------------------------------------------------------------ K4
// dL/dD[m] = g * (sum_n w_n e[n,m] / Z[m] + w_bg p_bg[m]).  Trimmed points (w == 0, bl.py:77) are
// compacted away while staging.  Single-chunk images store the final gradient; otherwise the raw
// chunk sum goes to gpart and bl_grad_reduce_kernel finishes.
template <int R, int C, bool POW2>
__device__ __forceinline__ bool bl_grad_body(const float2* __restrict__ pts_all, const int32_t* __restrict__ meta, int batch,
               const Geom& g, const Scale& k, int use_bg, int exact_cull, float inv_batch, const float* __restrict__ grad_loss,
               const float* __restrict__ amax_in, const float* __restrict__ rz_in,
               const float* __restrict__ pbg_in, const float* __restrict__ wsel,
               float* __restrict__ gpart, float* __restrict__ grad_density, int always_partial, const Xchg& x,
               unsigned int* __restrict__ tile_tick, int slot, int task) {
    __shared__ WarpTile<R> tiles[WARPS_PER_CTA];
    TaskInfo t;
    if (!decode_task<R, C>(meta, batch, g, t, slot, task)) return false;
    WarpTile<R>& tile = tiles[threadIdx.x >> 5];
    const size_t M = (size_t)g.hp * g.wp;
    const size_t img_base = (size_t)t.img * M;
    PixelTile<R, C> px;
    px.init(t, g);

    float acc[R][C], neg_amax[R][C];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            neg_amax[r][c] = __fmul_rn(-amax_in[img_base + px.pix(r, c)], LOG2E);
            acc[r][c] = 0.f;
        }

    const float2* pts = pts_all + t.pt_base;
    const float* w_pts = wsel + t.row0 + t.p_start;
    const ExpCull cull{exact_cull != 0, tile_max<R, C>(neg_amax), k.k1, px.box};
    const Scale2 k2s(k);
    f2 accp[R / 2][C], k2p[R / 2][C];
#pragma unroll
    for (int q = 0; q < R / 2; ++q)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            accp[q][c] = pack2(0.f, 0.f);
            k2p[q][c] = pack2(neg_amax[2 * q][c], neg_amax[2 * q + 1][c]);
        }
    constexpr bool PREFETCH = R * C < 16;
    float2 pf[PF];
    float pw[PF];
    if (PREFETCH && t.p_cnt > 0) fetch_points<true>(pts, w_pts, 0, t.p_cnt, pf, pw);
    for (int n0 = 0; n0 < t.p_cnt; n0 += TILE_PTS) {
        const int cnt = min(TILE_PTS, t.p_cnt - n0);
        __syncwarp();
        int kept;
        if (PREFETCH) {
            kept = stage_fetched_if<R>(tile, pf, pw, cnt, px.cym2, px.cyy,
                                       [&](float x, float y, float w) { return w != 0.f && cull.keep(x, y); });
            if (n0 + TILE_PTS < t.p_cnt) fetch_points<true>(pts, w_pts, n0 + TILE_PTS, t.p_cnt, pf, pw);
        } else {
            kept = stage_points_if<R, true, false>(
                tile, pts, w_pts, n0, cnt, px.cym2, px.cyy,
                [&](float x, float y, float w) { return w != 0.f && cull.keep(x, y); });
        }
        __syncwarp();
#pragma unroll 2
        for (int i = 0; i < kept; ++i) {
            const float w = tile.aux[i];
            const f2 w2 = pack2(w, w);
            const float2 xs = tile.xs[i];
            f2 yd[R / 2];
            load_yd2<R>(tile, i, yd);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float xd = axis_sqdist(xs.x, xs.y, px.cxm2[c], px.cxx[c]);
                const f2 xd2 = pack2(xd, xd);
#pragma unroll
                for (int q = 0; q < R / 2; ++q)
                    accp[q][c] = fma2(pair_exp2<POW2>(add2(yd[q], xd2), k2p[q][c], k2s), w2, accp[q][c]);
            }
        }
    }
#pragma unroll
    for (int q = 0; q < R / 2; ++q)
#pragma unroll
        for (int c = 0; c < C; ++c) unpack2(accp[q][c], acc[2 * q][c], acc[2 * q + 1][c]);

    if (!always_partial) {
        // One chunk: the sum is complete.  Several: park it in gpart; the task that arrives last at the tile adds the
        // chunk sums in chunk order and applies the per-pixel factors (no reduction kernel, no second pass).
        if (t.n_chunks > 1) {
            float* out = gpart + (size_t)t.chunk * M;
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int c = 0; c < C; ++c)
                    if (px.ok(r, c)) out[px.pix(r, c)] = acc[r][c];
            if (!tile_last_arrival(tile_tick + (size_t)t.img * g.tiles_img + t.task, t.n_chunks)) return false;
        }
        const float gscale = grad_loss[0] * inv_batch;
        const bool has_bg_row = use_bg || t.n_img_pts == 0;
        const float w_bg = has_bg_row ? wsel[t.row0 + t.n_rows - 1] : 0.f;
        // row-band sharding: the finished rows go straight into the workspace of the image's owner
        const unsigned int dst = x.peers ? x.mask[t.img] : 0u;
        float* gout = (dst ? xchg_ptr(x, __ffs(dst) - 1, x.region_off) : grad_density) + img_base;
        if (t.n_chunks > 1) {
            finish_grad_tile<R, C>(gpart + (size_t)t.first_chunk * M, t.n_chunks, M, t.row_base, t.col0, g.hp, g.wp, gscale, w_bg,
                                   rz_in + img_base, pbg_in + img_base, gout);
        } else {
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    if (!px.ok(r, c)) continue;
                    const int p = px.pix(r, c);
                    gout[p] = gscale * fmaf(acc[r][c], rz_in[img_base + p], w_bg * pbg_in[img_base + p]);
                }
        }
        return dst != 0u;
    } else {
        // sharded: chunks of an image finished by another rank go straight (and only) into that rank's workspace
        const unsigned int dst = x.peers ? x.mask[t.chunk] : 0u;
        float* out = (dst ? xchg_ptr(x, __ffs(dst) - 1, x.region_off) : gpart) + (size_t)t.chunk * M;
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int c = 0; c < C; ++c)
                if (px.ok(r, c)) out[px.pix(r, c)] = acc[r][c];
        return dst != 0u;
    }
}

template <int R, int C, bool POW2>
__global__ void __launch_bounds__(CTA_THREADS)
bl_grad_kernel(const float2* __restrict__ pts_all, const int32_t* __restrict__ meta, int batch, Geom g,
               Scale k, int use_bg, int exact_cull, float inv_batch, const float* __restrict__ grad_loss,
               const float* __restrict__ amax_in, const float* __restrict__ rz_in,
               const float* __restrict__ pbg_in, const float* __restrict__ wsel,
               float* __restrict__ gpart, float* __restrict__ grad_density, int always_partial, Xchg x,
               unsigned int* __restrict__ tile_tick, int n_slots, unsigned int* __restrict__ queue) {
    const int n_tiles = g.tiles - g.task_first;
    const unsigned int total = (unsigned)n_slots * (unsigned)n_tiles, first_round = gridDim.x * WARPS_PER_CTA;
    bool stored = false;
    for (unsigned int w = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5); w < total; w = queue_next_warp(queue, first_round)) {
        stored |= bl_grad_body<R, C, POW2>(pts_all, meta, batch, g, k, use_bg, exact_cull, inv_batch, grad_loss, amax_in, rz_in,
                                           pbg_in, wsel, gpart, grad_density, always_partial, x, tile_tick,
                                           (int)(w / n_tiles), g.task_first + (int)(w % n_tiles));
        __syncwarp();
    }
    queue_leave(queue);
    xchg_signal(x, stored);
}

// Multi-chunk images: add the chunk sums in chunk order and apply the per-pixel factors.
__device__ __forceinline__ bool bl_grad_reduce_body(const int32_t* __restrict__ meta, int batch, int M, int use_bg, float inv_batch,
                      const float* __restrict__ grad_loss, const float* __restrict__ gpart,
                      const float* __restrict__ rz_in, const float* __restrict__ pbg_in,
                      const float* __restrict__ wsel, float* __restrict__ grad_density, const Shard& sh, const Xchg& x,
                      int pix_first, int pix_end, int every_image);

__global__ void __launch_bounds__(256)
bl_grad_reduce_kernel(const int32_t* __restrict__ meta, int batch, int M, int use_bg, float inv_batch,
                      const float* __restrict__ grad_loss, const float* __restrict__ gpart,
                      const float* __restrict__ rz_in, const float* __restrict__ pbg_in,
                      const float* __restrict__ wsel, float* __restrict__ grad_density, Shard sh, Xchg x, int n_img,
                      int pix_first, int pix_end, int every_image) {
    xchg_wait(x);  // sharded: the gradient sums of the chunks other ranks swept
    bool stored = false;
    if ((int)blockIdx.y < n_img)
        stored = bl_grad_reduce_body(meta, batch, M, use_bg, inv_batch, grad_loss, gpart, rz_in, pbg_in, wsel, grad_density, sh, x,
                                     pix_first, pix_end, every_image);
    xchg_signal(x, stored);
}

__device__ __forceinline__ bool bl_grad_reduce_body(const int32_t* __restrict__ meta, int batch, int M, int use_bg, float inv_batch,
                      const float* __restrict__ grad_loss, const float* __restrict__ gpart,
                      const float* __restrict__ rz_in, const float* __restrict__ pbg_in,
                      const float* __restrict__ wsel, float* __restrict__ grad_density, const Shard& sh, const Xchg& x,
                      int pix_first, int pix_end, int every_image) {
    // pixels [pix_first, pix_end) of the image: all of them, or (row-band sharding) the rank's band of grid rows
    const int img = sh.img_lo + blockIdx.y;
    const Meta mv = meta_view(meta, batch);
    const int first = mv.icb[img], n_chunks = mv.icb[img + 1] - first;
    if (sh.on) {  // every image is finished by the rank that owns its first chunk, single-chunk images included
        if (first < sh.chunk_lo || first >= sh.chunk_hi) return false;
    } else if (n_chunks <= 1 && !every_image) {
        return false;
    }
    const int pix = pix_first + blockIdx.x * 256 + threadIdx.x;
    if (pix >= pix_end) return false;
    float acc = 0.f;
    for (int c = 0; c < n_chunks; ++c) acc += gpart[(size_t)(first + c) * M + pix];
    const int n_rows = mv.row_off[img + 1] - mv.row_off[img];
    const bool has_bg_row = use_bg || mv.pt_off[img + 1] == mv.pt_off[img];
    const float w_bg = has_bg_row ? wsel[mv.row_off[img] + n_rows - 1] : 0.f;
    const size_t m = (size_t)img * M + pix;
    const float gv = grad_loss[0] * inv_batch * fmaf(acc, rz_in[m], w_bg * pbg_in[m]);
    const unsigned int dst = x.peers ? x.mask[img] : 0u;  // the image's owner, when that is another rank
    if (dst) xchg_store(x, dst, x.region_off, m, gv);
    else grad_density[m] = gv;
    return dst != 0u;
}

// ------------------------------------------------------------------------- posterior (API parity)
// rz / pbg from the chunk shares (the fused forward gets them as a by-product of bl_counts_kernel).
__global__ void __launch_bounds__(256)
bl_finish_z_kernel(const int32_t* __restrict__ meta, int batch, int M, const float* __restrict__ zpart,
                   const float* __restrict__ ebg_in, float* __restrict__ rz_out, float* __restrict__ pbg_out,
                   int img_first, Xchg x, int n_img) {
    xchg_wait(x);  // sharded: the other ranks' denominator shares (and the density, for the kernel that follows)
    if ((int)blockIdx.y >= n_img) return;
    const int img = img_first + blockIdx.y;
    const Meta mv = meta_view(meta, batch);
    const int pix = blockIdx.x * 256 + threadIdx.x;
    if (pix >= M) return;
    const size_t m = (size_t)img * M + pix;
    const float ebg = ebg_in[m];
    const float rz = softmax_rz(zpart, (size_t)M, mv.icb[img], mv.icb[img + 1] - mv.icb[img], pix, ebg);
    rz_out[m] = rz;
    pbg_out[m] = ebg * rz;
}

template <int R, int C, bool POW2>
__global__ void __launch_bounds__(CTA_THREADS)
bl_posterior_kernel(const float2* __restrict__ pts_all, const int32_t* __restrict__ meta, int batch, Geom g,
                    Scale k, int use_bg, const float* __restrict__ amax_in, const float* __restrict__ rz_in,
                    const float* __restrict__ pbg_in, float* __restrict__ prob_out) {
    __shared__ WarpTile<R> tiles[WARPS_PER_CTA];
    TaskInfo t;
    if (!decode_task<R, C>(meta, batch, g, t, blockIdx.y, g.task_first + blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5))) return;
    WarpTile<R>& tile = tiles[threadIdx.x >> 5];
    const size_t M = (size_t)g.hp * g.wp;
    const size_t img_base = (size_t)t.img * M;
    PixelTile<R, C> px;
    px.init(t, g);
    float* prob = prob_out + (size_t)t.row0 * M;

    float neg_amax[R][C], rz[R][C];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int p = px.pix(r, c);
            neg_amax[r][c] = __fmul_rn(-amax_in[img_base + p], LOG2E);
            rz[r][c] = rz_in[img_base + p];
            if (px.ok(r, c) && t.chunk == t.first_chunk && (use_bg || t.n_img_pts == 0))
                prob[(size_t)(t.n_rows - 1) * M + p] = pbg_in[img_base + p];
        }
    const float2* pts = pts_all + t.pt_base;
    prob += (size_t)t.p_start * M;
    for (int n0 = 0; n0 < t.p_cnt; n0 += TILE_PTS) {
        const int cnt = min(TILE_PTS, t.p_cnt - n0);
        __syncwarp();
        stage_points<R>(tile, pts, n0, t.p_cnt, cnt, px.cym2, px.cyy);
        __syncwarp();
#pragma unroll 1
        for (int i = 0; i < cnt; ++i) {
            const float2 xs = tile.xs[i];
            float yd[R];
            load_yd<R>(tile, i, yd);
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float xd = axis_sqdist(xs.x, xs.y, px.cxm2[c], px.cxx[c]);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const float p = pair_exp<POW2>(__fadd_rn(yd[r], xd), neg_amax[r][c], k) * rz[r][c];
                    if (px.ok(r, c)) prob[(size_t)(n0 + i) * M + px.pix(r, c)] = p;
                }
            }
        }
    }
}

// ------------------------------------------------------- Bay_Loss on materialised posteriors
// counts[row] = sum_m D[m] * prob[row, m]: one warp per row, coalesced, fixed order.
__global__ void __launch_bounds__(256)
bl_prob_counts_kernel(const float* __restrict__ prob, const float* __restrict__ density,
                      const int32_t* __restrict__ meta, int batch, int M, int64_t total_rows,
                      float* __restrict__ cpart, unsigned int* __restrict__ ticket) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *ticket = 0u;  // bl_select_kernel's arrival counter
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= total_rows) return;
    const int lane = threadIdx.x & 31;
    const int32_t* row_off = meta + (batch + 1);
    int img = 0;
    while (img + 1 < batch && row >= row_off[img + 1]) ++img;
    const float* d = density + (size_t)img * M;
    const float* p = prob + (size_t)row * M;
    float s = 0.f;
    for (int m = lane; m < M; m += 32) s = fmaf(d[m], p[m], s);
    s = warp_sum(s);
    if (lane == 0) cpart[row] = s;
}

// grad[b,m] = g * sum_rows w[row] * prob[row,m]
__global__ void __launch_bounds__(256)
bl_prob_grad_kernel(const float* __restrict__ prob, const int32_t* __restrict__ meta, int batch, int M,
                    float inv_batch, const float* __restrict__ grad_loss, const float* __restrict__ wsel,
                    float* __restrict__ grad_density) {
    const int img = blockIdx.y;
    const int m = blockIdx.x * 256 + threadIdx.x;
    if (m >= M) return;
    const int32_t* row_off = meta + (batch + 1);
    const int r0 = row_off[img], r1 = row_off[img + 1];
    float acc = 0.f;
    for (int r = r0; r < r1; ++r) {
        const float w = wsel[r];
        if (w != 0.f) acc = fmaf(w, prob[(size_t)r * M + m], acc);
    }
    grad_density[(size_t)img * M + m] = grad_loss[0] * inv_batch * acc;
}

// ------------------------------------------------------------------- point-chunk sharding across GPUs
// One batch spread over the GPUs of a box by POINT CHUNKS (dgvcc_bl_shard_*): every rank sweeps its own chunks over
// all pixels of the images they belong to; the per-chunk partials an image's other ranks need (minima, denominator
// shares, gradient sums), the counts / residuals of its rows, the density and the finished gradient travel as plain
// stores into the peers' workspaces over NVLink (peer pointers from dgvcc_peer_open), followed by a flag per
// (phase, source rank).  Receivers combine the partials in chunk order, exactly like one GPU does, so the sharded
// result is bit-identical to the single-GPU one.  No NCCL on the data path.
constexpr int PUSH_THREADS = 256;

// One CTA per slice: copy `bytes` from src_base + src_off to peers[dst_rank] + dst_off.  The last CTA to finish
// raises this rank's flag of `phase` on every rank in signal_mask (release at system scope, after every CTA's
// stores were fenced), so a receiver that sees the flag sees the data.
__global__ void __launch_bounds__(PUSH_THREADS)
bl_push_kernel(const dgvcc_bl_push* __restrict__ slices, int n_slices, const char* __restrict__ src_base,
               char* const* __restrict__ peers, int64_t flags_off, int phase, int rank, int world,
               unsigned int signal_mask, unsigned int epoch, unsigned int* __restrict__ ticket) {
    __shared__ bool last;
    if ((int)blockIdx.x < n_slices) {
        const dgvcc_bl_push sl = slices[blockIdx.x];
        const char* src = src_base + sl.src_off;
        char* dst = peers[sl.dst_rank] + sl.dst_off;
        if ((((uintptr_t)src | (uintptr_t)dst | (uintptr_t)sl.bytes) & 15u) == 0) {
            const int n = sl.bytes >> 4;
            for (int i = threadIdx.x; i < n; i += PUSH_THREADS)
                reinterpret_cast<int4*>(dst)[i] = __ldcg(reinterpret_cast<const int4*>(src) + i);
        } else {
            const int n = sl.bytes >> 2;  // every region is made of 4-byte elements
            for (int i = threadIdx.x; i < n; i += PUSH_THREADS)
                reinterpret_cast<int*>(dst)[i] = __ldcg(reinterpret_cast<const int*>(src) + i);
        }
    }
    fence_acq_rel_gpu();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    fence_acq_rel_gpu();
    if ((int)threadIdx.x < world && ((signal_mask >> threadIdx.x) & 1u)) {
        unsigned int* flag = reinterpret_cast<unsigned int*>(peers[threadIdx.x] + flags_off) + phase * world + rank;
        st_release_sys(flag, epoch);
    }
    if (threadIdx.x == 0) *ticket = 0u;
}

// A rank without work in a phase still raises its flag.
__global__ void bl_signal_kernel(Xchg x) { xchg_signal(x); }

// Local variant: the same slices with one destination base and no flags (gathers a rank's own finished gradients).
__global__ void __launch_bounds__(PUSH_THREADS)
bl_copy_kernel(const dgvcc_bl_push* __restrict__ slices, int n_slices, const char* __restrict__ src_base,
               char* __restrict__ dst_base, Xchg x) {
    xchg_wait(x);  // the finished gradients other ranks delivered
    if ((int)blockIdx.x >= n_slices) return;
    const dgvcc_bl_push sl = slices[blockIdx.x];
    const char* src = src_base + sl.src_off;
    char* dst = dst_base + sl.dst_off;
    if ((((uintptr_t)src | (uintptr_t)dst | (uintptr_t)sl.bytes) & 15u) == 0) {
        for (int i = threadIdx.x; i < (sl.bytes >> 4); i += PUSH_THREADS)
            reinterpret_cast<int4*>(dst)[i] = __ldcg(reinterpret_cast<const int4*>(src) + i);
    } else {
        for (int i = threadIdx.x; i < (sl.bytes >> 2); i += PUSH_THREADS)
            reinterpret_cast<int*>(dst)[i] = __ldcg(reinterpret_cast<const int*>(src) + i);
    }
}

// Wait until every rank in wait_mask has raised its flag of this phase to `epoch` (lane = source rank).  Bounded:
// after `timeout_ns` the kernel records the phase in err[0] and returns, so a lost peer cannot hang the GPU.
__global__ void __launch_bounds__(32)
bl_wait_kernel(const unsigned int* __restrict__ flags, int phase, int world, unsigned int wait_mask,
               unsigned int epoch, unsigned long long timeout_ns, int* __restrict__ err) {
    const int src = threadIdx.x;
    if (src < world && ((wait_mask >> src) & 1u)) {
        const unsigned int* flag = flags + phase * world + src;
        const unsigned long long t0 = global_ns();
        while ((int)(ld_acquire_sys(flag) - epoch) < 0) {
            if (global_ns() - t0 > timeout_ns) {
                atomicExch(err, 1 + phase + 16 * src);
                break;
            }
            __nanosleep(64);
        }
    }
}

// Sum of the per-image losses in image order (every rank received the values of the images it does not hold).
__global__ void bl_loss_finish_kernel(const float* __restrict__ loss_img, int batch, float inv_batch,
                                      float* __restrict__ loss_out, Xchg x) {
    xchg_wait(x);
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        float total = 0.f;
        const volatile float* li = loss_img;  // written by the peers
        for (int i = 0; i < batch; ++i) total += li[i];
        loss_out[0] = total * inv_batch;
    }
}

// ------------------------------------------------------------------- row-band sharding across GPUs
// One batch spread over the GPUs of a box by PIXELS (dgvcc_bl_band_*): rank r sweeps ALL points of every image over
// its own band of grid rows.  The softmax of bl.py:44 runs over the points of ONE pixel, so minima, denominators,
// posteriors and the density gradient of a pixel never leave the rank that owns it; only the expected counts of
// bl.py:73 are sums over pixels.  bl_counts_kernel stores the per-CTA partial counts of the band on every rank as it
// produces them; every rank then adds all partial rows in pixel-tile order (the same bits everywhere, and the same sum
// as on one GPU) and finds the top-k cut and the loss for itself.  One data-dependent exchange per step (CNT) against
// four for the point-chunk split; DENS (owner -> band ranks) hides on a side stream, GRAD (band -> owner, stored by
// bl_grad_kernel itself) ends the step.

// Partial-count rows per rank in the count-share table (the bands follow from the grid shape and the world size).
struct BandRows { int n[32]; };

// Expected counts = all partial rows added in (rank, CTA) order, i.e. in the order of the pixel tiles -- with bands cut
// at CTA boundaries exactly the sum bl_reduce_counts_kernel forms on one GPU; residual |t - c| (bl.py:73-75).  Every rank
// runs this over all rows of the batch and gets the same bits.
__global__ void __launch_bounds__(256)
bl_band_combine_kernel(const float* __restrict__ cshare, int world, int share_rows, BandRows rows, int64_t total_rows,
                       const int32_t* __restrict__ meta, const float* __restrict__ targets, int batch,
                       float* __restrict__ counts, float* __restrict__ residual, Xchg x) {
    xchg_wait(x);  // the partial rows of the other ranks
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= total_rows) return;
    float c = 0.f;
    for (int q = 0; q < world; ++q) {
        const float* p = cshare + (size_t)q * share_rows * total_rows + j;
#pragma unroll 4
        for (int tl = 0; tl < rows.n[q]; ++tl) c += __ldcg(p + (size_t)tl * total_rows);
    }
    const Meta mv = meta_view(meta, batch);
    int lo = 0, hi = batch;  // image of row j
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (mv.row_off[mid] <= j) lo = mid; else hi = mid;
    }
    const int local = (int)(j - mv.row_off[lo]);
    const int n_pts = mv.pt_off[lo + 1] - mv.pt_off[lo];
    const float tgt = (local < n_pts) ? targets[mv.pt_off[lo] + local] : 0.f;
    counts[j] = c;
    residual[j] = fabsf(__fadd_rn(tgt, -c));
}

// ------------------------------------------------------------------------------- host side
static bool is_pow2(float s) {
    int e;
    return s > 0.f && frexpf(s, &e) == 0.5f;
}

static Scale make_scale(float sigma) {
    Scale k;
    k.s = (float)(2.0 * (double)sigma * (double)sigma);  // python: 2.0 * sigma ** 2, then cast to fp32
    k.r = 1.0f / k.s;
    k.neg_inv_s = -k.r;
    k.k1 = (float)(-1.4426950408889634 / (double)k.s);
    return k;
}

// Pixel tile per thread (rows x columns): the largest one that still yields ~16 warp tasks per SM.
// More pixels per thread = fewer LDS per exponential (the kernels are bound by the MIO path).
struct Variant { int rows, cols; };
static const Variant kVariants[] = {{8, 2}, {8, 1}, {4, 1}, {2, 1}};

static long variant_tasks(const Variant& v, int total_chunks, int hp, int wp) {
    return (long)total_chunks * ceil_div(wp, 32 * v.cols) * ceil_div(hp, v.rows);
}

// Tuning knobs of benchmarks and experiments (dgvcc_bl_set_option): host-side, read when a plan is made.
static int g_opt_min_cell = 64;   // smallest cell of the point grid of the minima, image pixels (a power of two)
static int g_opt_band_tile = 0;   // pixel tile of the symmetric (sharded) layouts: 0 = by task count, else rows*10 + cols

static Variant pick_variant(int total_chunks, int hp, int wp) {
    const long want = 148L * 16;
    for (const Variant& v : kVariants)
        if (variant_tasks(v, total_chunks, hp, wp) >= want) return v;
    return kVariants[3];
}

static Geom make_geom(int hp, int wp, const Variant& v, float stride) {
    Geom g;
    g.hp = hp; g.wp = wp;
    g.col_blocks = ceil_div(wp, 32 * v.cols);
    g.tiles = g.col_blocks * ceil_div(hp, v.rows);
    g.task_first = 0;
    g.tiles_img = g.tiles;
    g.stride = stride;
    g.half = stride / 2.0f;
    return g;
}

static int layout(int64_t total_rows, int total_chunks, int batch, int hp, int wp, dgvcc_bl_layout* L, int world = 0) {
    if (!L || total_rows < batch || total_chunks < batch || batch <= 0 || hp <= 0 || wp <= 0 || world < 0 || world > 32)
        return DGVCC_ERR_ARG;
    // world > 0: the symmetric layout of dgvcc_bl_shard_* (identical on every rank); the pixel tile is chosen for the
    // chunks ONE rank sweeps
    Variant v = pick_variant(world > 0 ? ceil_div(total_chunks, world) : total_chunks, hp, wp);
    // A rank of a sharded sweep has about one round of warp tasks: the 8 x 32 tile (twice the tasks, half as long) balances
    // better than 8 x 64 -- measured on 2 and 8 B200 with config 3 (profiles/r2_strong_scaling.md), 3-7 % of the step.
    if (world > 1 && v.rows == 8 && v.cols == 2) v = kVariants[1];
    if (world > 0 && g_opt_band_tile) v = Variant{g_opt_band_tile / 10, g_opt_band_tile % 10};
    const int tiles = make_geom(hp, wp, v, 1.f).tiles;
    const size_t M = (size_t)hp * wp;
    const size_t pix = (size_t)batch * M * sizeof(float);
    const size_t rows = (size_t)total_rows * sizeof(float);
    const size_t chunk_pix = (size_t)total_chunks * M * sizeof(float);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return (int64_t)o; };
    L->dens = L->gfinal = L->flags = L->err = L->push_ticket = L->cshare = 0;
    L->share_rows = 0;
    if (world > 0) {  // fixed offsets, whatever the batch: the flags outlive a step (they are compared with the epoch)
        L->flags = take((size_t)DGVCC_BL_PHASES * 32 * sizeof(unsigned int));
        L->err = take(sizeof(int));
        L->push_ticket = take(2 * sizeof(unsigned int));  // [0] fused producers (main stream), [1] the DENS copy (side stream)
    }
    L->amax = take(pix); L->rz = take(pix); L->pbg = take(pix); L->ebg = take(pix);
    L->counts = take(rows); L->wsel = take(rows); L->residual = take(rows);
    L->loss_img = take((size_t)batch * sizeof(float));
    L->ticket = take(sizeof(unsigned int));
    const int count_rows = ceil_div(tiles, WARPS_PER_CTA);  // one partial row per CTA of bl_counts_kernel
    L->cpart = take((size_t)count_rows * rows);
    L->zpart = take(chunk_pix);
    L->gpart = take(chunk_pix);
    L->minpart = L->gpart;       // (no per-chunk minima any more: bl_gridmin_kernel writes per-image minima into the pbg region)
    L->goff = take((size_t)batch * (GRID_MAX_CELLS + 1) * sizeof(int32_t));   // grid cell offsets per image
    L->gsorted = take((size_t)total_rows * sizeof(float2));                   // points sorted by grid cell (<= rows)
    L->ztick = take((size_t)batch * tiles * sizeof(unsigned int));            // arrival counters per (image, pixel tile): bl_z
    L->gtick = take((size_t)batch * tiles * sizeof(unsigned int));            //                                          bl_grad
    L->queue = take(6 * sizeof(unsigned int));   // work queues of the persistent sweeps: (handed out, CTAs gone) x z, counts, grad
    if (world > 0) {
        L->dens = take(pix);         // density of every image this rank sweeps, delivered by the image's owner
        L->gfinal = take(pix);       // finished gradients, delivered to the image's owner
        // row-band sharding: the per-CTA partial counts of every rank's band (bl_counts_kernel stores them on every rank)
        const int band_tile_rows = ceil_div(ceil_div(hp, v.rows), world);
        L->share_rows = ceil_div(band_tile_rows * make_geom(hp, wp, v, 1.f).col_blocks, WARPS_PER_CTA);
        L->cshare = take((size_t)world * L->share_rows * rows);
    }
    L->total = (int64_t)off;
    L->tiles = count_rows;
    L->rows_per_thread = v.rows;
    L->cols_per_thread = v.cols;
    return DGVCC_OK;
}

template <typename T>
static T* at(const void* ws, int64_t off) { return reinterpret_cast<T*>((char*)ws + off); }

}  // namespace bl
}  // namespace dgvcc

using namespace dgvcc;
using namespace dgvcc::bl;

extern "C" int dgvcc_abi_version(void) { return 10; }
extern "C" int dgvcc_bounds_checked(void) { return DGVCC_BOUNDS_CHECKED; }

extern "C" int dgvcc_bl_workspace_layout(int64_t total_rows, int total_chunks, int batch, int hp, int wp,
                                         dgvcc_bl_layout* out) {
    return layout(total_rows, total_chunks, batch, hp, wp, out);
}

// KERNEL<R, C, POW2> for the (rows, cols) variant chosen by pick_variant()
#define BL_LAUNCH_RC(R_, C_, POW2_, KERNEL, GRID, STREAM, ...)                              \
    do {                                                                                    \
        if (POW2_) KERNEL<R_, C_, true><<<GRID, CTA_THREADS, 0, STREAM>>>(__VA_ARGS__);     \
        else KERNEL<R_, C_, false><<<GRID, CTA_THREADS, 0, STREAM>>>(__VA_ARGS__);          \
    } while (0)
#define BL_DISPATCH(V_, POW2_, KERNEL, GRID, STREAM, ...)                                              \
    do {                                                                                               \
        if ((V_).rows == 8 && (V_).cols == 2) BL_LAUNCH_RC(8, 2, POW2_, KERNEL, GRID, STREAM, __VA_ARGS__); \
        else if ((V_).rows == 8) BL_LAUNCH_RC(8, 1, POW2_, KERNEL, GRID, STREAM, __VA_ARGS__);         \
        else if ((V_).rows == 4) BL_LAUNCH_RC(4, 1, POW2_, KERNEL, GRID, STREAM, __VA_ARGS__);         \
        else BL_LAUNCH_RC(2, 1, POW2_, KERNEL, GRID, STREAM, __VA_ARGS__);                             \
    } while (0)

// Persistent launch: at most as many CTAs as the GPU holds at once (occupancy of this very instantiation, asked once
// per kernel and device); the kernel's work queue hands out the rest of the items.
static int resident_ctas(const void* key, int per_sm_query(int*)) {
    struct Entry { const void* key; int dev, ctas; };
    static Entry cache[256];
    static int n_cached = 0;
    static std::mutex mu;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 1;
    std::lock_guard<std::mutex> lock(mu);
    for (int i = 0; i < n_cached; ++i)
        if (cache[i].key == key && cache[i].dev == dev) return cache[i].ctas;
    int per_sm = 0, sms = 0;
    if (per_sm_query(&per_sm) != 0 || per_sm < 1) per_sm = 1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1) sms = 1;
    if (n_cached < 256) cache[n_cached++] = Entry{key, dev, per_sm * sms};
    return per_sm * sms;
}
#define BL_PERSIST_ONE(KERNEL_INST, WANTED, STREAM, ...)                                                              \
    do {                                                                                                              \
        auto kern_ = KERNEL_INST;                                                                                     \
        const int cap_ = resident_ctas((const void*)kern_, [](int* n) {                                               \
            return (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(n, KERNEL_INST, CTA_THREADS, 0); });            \
        const int grid_ = (WANTED) < cap_ ? (WANTED) : cap_;                                                          \
        kern_<<<grid_ > 0 ? grid_ : 1, CTA_THREADS, 0, STREAM>>>(__VA_ARGS__);                                        \
    } while (0)
#define BL_PERSIST_RC(R_, C_, POW2_, KERNEL, WANTED, STREAM, ...)                                    \
    do {                                                                                             \
        if (POW2_) BL_PERSIST_ONE((KERNEL<R_, C_, true>), WANTED, STREAM, __VA_ARGS__);              \
        else BL_PERSIST_ONE((KERNEL<R_, C_, false>), WANTED, STREAM, __VA_ARGS__);                   \
    } while (0)
#define BL_PERSIST(V_, POW2_, KERNEL, WANTED, STREAM, ...)                                                    \
    do {                                                                                                      \
        if ((V_).rows == 8 && (V_).cols == 2) BL_PERSIST_RC(8, 2, POW2_, KERNEL, WANTED, STREAM, __VA_ARGS__); \
        else if ((V_).rows == 8) BL_PERSIST_RC(8, 1, POW2_, KERNEL, WANTED, STREAM, __VA_ARGS__);             \
        else if ((V_).rows == 4) BL_PERSIST_RC(4, 1, POW2_, KERNEL, WANTED, STREAM, __VA_ARGS__);             \
        else BL_PERSIST_RC(2, 1, POW2_, KERNEL, WANTED, STREAM, __VA_ARGS__);                                 \
    } while (0)

extern "C" int dgvcc_bl_set_option(int option, int value) {
    switch (option) {
        case DGVCC_BL_OPT_MIN_CELL:
            if (value < 8 || value > 4096 || (value & (value - 1))) return DGVCC_ERR_ARG;
            g_opt_min_cell = value;
            return DGVCC_OK;
        case DGVCC_BL_OPT_BAND_TILE:
            if (value != 0 && value != 82 && value != 81 && value != 41 && value != 21) return DGVCC_ERR_ARG;
            g_opt_band_tile = value;
            return DGVCC_OK;
        default:
            return DGVCC_ERR_ARG;
    }
}

namespace {

struct Plan {
    dgvcc_bl_layout L;
    Geom g;
    Scale k;
    Variant v;
    bool pow2;
    dim3 grid;   // (CTAs per chunk, chunks this launch sweeps)
    Shard sh;
    // CTAs that hold every warp task of bl_z / bl_grad at once (the persistent launches take fewer when the GPU is full)
    int warp_ctas() const { return ceil_div((int)grid.y * (g.tiles - g.task_first), WARPS_PER_CTA); }
};

// What every plan starts from (world > 0: the symmetric layout of the sharded paths); the callers add checks and grid.
int plan_common(const void* a, const void* ws, size_t ws_bytes, int batch, int hp, int wp, int64_t total_rows,
                int total_chunks, float stride, float sigma, int world, Plan* p) {
    if (!a || !ws) return DGVCC_ERR_ARG;
    if (!(stride > 0.f) || !(sigma > 0.f)) return DGVCC_ERR_ARG;
    int rc = layout(total_rows, total_chunks, batch, hp, wp, &p->L, world);
    if (rc) return rc;
    if (ws_bytes < (size_t)p->L.total) return DGVCC_ERR_WORKSPACE;
    p->v = Variant{p->L.rows_per_thread, p->L.cols_per_thread};
    p->g = make_geom(hp, wp, p->v, stride);
    p->k = make_scale(sigma);
    p->pow2 = is_pow2(p->k.s);
    p->sh = no_shard();
    return DGVCC_OK;
}

int make_plan(const void* a, const void* b, const void* ws, size_t ws_bytes, int batch, int hp, int wp,
              int64_t total_rows, int total_chunks, float stride, float sigma, Plan* p,
              const dgvcc_bl_shard* shard = nullptr) {
    if (!b) return DGVCC_ERR_ARG;
    int rc = plan_common(a, ws, ws_bytes, batch, hp, wp, total_rows, total_chunks, stride, sigma, shard ? shard->world : 0, p);
    if (rc) return rc;
    int slots = total_chunks;
    if (shard) {
        if (shard->world < 1 || shard->rank < 0 || shard->rank >= shard->world || shard->chunk_lo < 0 ||
            shard->chunk_hi < shard->chunk_lo || shard->chunk_hi > total_chunks || shard->img_lo < 0 ||
            shard->img_hi < shard->img_lo || shard->img_hi > batch)
            return DGVCC_ERR_ARG;
        p->sh = Shard{1, shard->chunk_lo, shard->chunk_hi, shard->pt_lo, shard->pt_hi, shard->img_lo, shard->img_hi};
        slots = shard->chunk_hi - shard->chunk_lo;
    }
    p->grid = dim3(ceil_div(p->g.tiles, WARPS_PER_CTA), slots);
    return DGVCC_OK;
}

inline void mark(void** events, int i, cudaStream_t st) {
    if (events && events[i]) cudaEventRecord((cudaEvent_t)events[i], st);
}

GridGeom make_grid(int hp, int wp, float stride) {
    const float ex = wp * stride, ey = hp * stride;
    GridGeom gg;
    gg.cell = (float)g_opt_min_cell;
    for (;;) {
        gg.gx = (int)ceilf(ex / gg.cell);
        gg.gy = (int)ceilf(ey / gg.cell);
        if ((long)gg.gx * gg.gy <= GRID_MAX_CELLS) break;
        gg.cell *= 2.f;
    }
    gg.gx = gg.gx < 1 ? 1 : gg.gx;
    gg.gy = gg.gy < 1 ? 1 : gg.gy;
    gg.inv_cell = 1.f / gg.cell;
    const float e = ex > ey ? ex : ey;
    gg.slack_m = 32.f * e * e;   // covers points up to four grid extents away; farther ones are far beyond any bound
    return gg;
}

// per-pixel minima of the images [img_first, img_first + n_img): grid build + ring walk, into min_img [B, hp*wp]
int launch_gridmin(const Plan& p, const float2* pts, const int32_t* meta, int batch, int hp, int wp, int img_first, int n_img,
                   void* ws, float* min_img, cudaStream_t st, int row_lo = 0, int row_hi = -1) {
    if (row_hi < 0) row_hi = hp;   // grid rows [row_lo, row_hi) of every image (row_lo even): the whole grid, or a rank's band
    if (n_img <= 0 || row_hi <= row_lo) return DGVCC_OK;
    const GridGeom gg = make_grid(hp, wp, p.g.stride);
    int32_t* goff = at<int32_t>(ws, p.L.goff);
    float2* gsorted = at<float2>(ws, p.L.gsorted);
    bl_grid_build_kernel<<<n_img, 1024, 0, st>>>(pts, meta, batch, gg, img_first, goff, gsorted, at<unsigned int>(ws, p.L.ztick),
                                                 at<unsigned int>(ws, p.L.gtick), p.g.tiles_img, at<unsigned int>(ws, p.L.queue));
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    // The minima have their own, small pixel tile (2 rows x 32 columns), independent of the exponential sweeps': every point
    // inside a tile's own rectangle is swept over the whole tile whatever the bound, so a crowd of 1500 heads inside one
    // 8 x 64 tile is a 50k-instruction warp -- the critical path of the launch.  Measured on the config-3 batch (grid
    // build included): 8x2 123 us, 8x1 85, 4x1 75, 2x1 70.
    const Variant v{2, 1};
    Geom gm = make_geom(hp, wp, v, p.g.stride);
    gm.task_first = (row_lo / v.rows) * gm.col_blocks;
    gm.tiles = ceil_div(row_hi, v.rows) * gm.col_blocks;
    const dim3 grid(ceil_div(gm.tiles - gm.task_first, WARPS_PER_CTA), n_img);
    bl_gridmin_kernel<2, 1><<<grid, CTA_THREADS, 0, st>>>(gsorted, goff, meta, batch, gm, gg, img_first, min_img);
    return (int)cudaGetLastError();
}

// partial minima (multi-chunk images only) + softmax max / denominator shares
int launch_z(const Plan& p, const float* pts_xy, const int32_t* meta, const float* st_sizes, int batch,
             int multi_chunk, float bg_ratio, int use_bg, int exact_cull, void* ws, cudaStream_t st,
             void** events = nullptr) {
    float* min_img = at<float>(ws, p.L.gpart);   // free until the backward pass (bl_z_kernel's last arrivals write rz / pbg)
    const float2* pts = (const float2*)pts_xy;
    (void)multi_chunk;
    mark(events, 0, st);
    int rc = launch_gridmin(p, pts, meta, batch, p.g.hp, p.g.wp, 0, batch, ws, min_img, st);
    if (rc) return rc;
    mark(events, 1, st);
    BL_PERSIST(p.v, p.pow2, bl_z_kernel, p.warp_ctas(), st, pts, meta, st_sizes, batch, p.g, p.k, bg_ratio, use_bg,
                exact_cull, at<float>(ws, p.L.zpart), at<float>(ws, p.L.amax), at<float>(ws, p.L.ebg),
                at<unsigned int>(ws, p.L.ticket), p.sh, (const float*)min_img, Xchg{}, at<float>(ws, p.L.rz),
                at<float>(ws, p.L.pbg), at<unsigned int>(ws, p.L.ztick), 1, (int)p.grid.y, at<unsigned int>(ws, p.L.queue) + 0);
    mark(events, 2, st);
    return (int)cudaGetLastError();
}

int launch_reduce_counts(const dgvcc_bl_layout& L, const float* targets, const int32_t* meta, int batch,
                         int64_t total_rows, int tiles, void* ws, const Shard& sh, cudaStream_t st) {
    bl_reduce_counts_kernel<<<(unsigned)((total_rows + 255) / 256), 256, 0, st>>>(
        at<float>(ws, L.cpart), tiles, total_rows, meta, targets, batch, at<float>(ws, L.counts),
        at<float>(ws, L.residual), sh, Xchg{}, (int64_t)0);
    return (int)cudaGetLastError();
}

int launch_select(const dgvcc_bl_layout& L, const float* targets, const int32_t* meta, int batch,
                  int64_t total_rows, float inv_batch, int tiles, void* ws, float* loss_out, cudaStream_t st) {
    int rc = launch_reduce_counts(L, targets, meta, batch, total_rows, tiles, ws, no_shard(), st);
    if (rc) return rc;
    bl_select_kernel<<<batch, SELECT_THREADS, 0, st>>>(
        meta, targets, batch, inv_batch, at<float>(ws, L.counts), at<float>(ws, L.residual), at<float>(ws, L.wsel),
        at<float>(ws, L.loss_img), loss_out, at<unsigned int>(ws, L.ticket), 0, 1, no_shard(), Xchg{}, batch);
    return (int)cudaGetLastError();
}

}  // namespace

extern "C" int dgvcc_bl_forward_profiled(const float* pts_xy, const float* targets, const int32_t* meta,
                                         const float* st_sizes, const float* density, int batch, int hp, int wp,
                                         int64_t total_rows, int total_chunks, int multi_chunk, float stride,
                                         float sigma, float bg_ratio, int use_bg, int exact_cull, float inv_batch,
                                         void* workspace, size_t workspace_bytes, float* loss_out, void* stream,
                                         void** events) {
    DGVCC_DEVICE_GUARD(stream);
    Plan p;
    int rc = make_plan(meta, density, workspace, workspace_bytes, batch, hp, wp, total_rows, total_chunks, stride,
                       sigma, &p);
    if (rc) return rc;
    if (!st_sizes || !loss_out || !pts_xy || !targets) return DGVCC_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = launch_z(p, pts_xy, meta, st_sizes, batch, multi_chunk, bg_ratio, use_bg, exact_cull, workspace, st, events))) return rc;
    BL_PERSIST(p.v, p.pow2, bl_counts_kernel, (int)(p.grid.x * p.grid.y), st, (const float2*)pts_xy, meta, density, batch, p.g, p.k,
                use_bg, exact_cull, at<float>(workspace, p.L.amax), at<float>(workspace, p.L.rz), at<float>(workspace, p.L.pbg),
                total_rows, at<float>(workspace, p.L.cpart), -1, Xchg{}, (int)p.grid.y, at<unsigned int>(workspace, p.L.queue) + 2);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    mark(events, 3, st);
    rc = launch_select(p.L, targets, meta, batch, total_rows, inv_batch, p.L.tiles, workspace, loss_out, st);
    mark(events, 4, st);
    return rc;
}

extern "C" int dgvcc_bl_forward(const float* pts_xy, const float* targets, const int32_t* meta,
                                const float* st_sizes, const float* density, int batch, int hp, int wp,
                                int64_t total_rows, int total_chunks, int multi_chunk, float stride, float sigma,
                                float bg_ratio, int use_bg, int exact_cull, float inv_batch, void* workspace,
                                size_t workspace_bytes, float* loss_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    return dgvcc_bl_forward_profiled(pts_xy, targets, meta, st_sizes, density, batch, hp, wp, total_rows,
                                     total_chunks, multi_chunk, stride, sigma, bg_ratio, use_bg, exact_cull,
                                     inv_batch, workspace, workspace_bytes, loss_out, stream, nullptr);
}

extern "C" int dgvcc_bl_backward(const float* pts_xy, const int32_t* meta, int batch, int hp, int wp,
                                 int64_t total_rows, int total_chunks, int multi_chunk, float stride, float sigma,
                                 int use_bg, int exact_cull, float inv_batch, const float* grad_loss,
                                 void* workspace, size_t workspace_bytes, float* grad_density, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    Plan p;
    int rc = make_plan(meta, grad_loss, workspace, workspace_bytes, batch, hp, wp, total_rows, total_chunks, stride,
                       sigma, &p);
    if (rc) return rc;
    if (!grad_density || !pts_xy) return DGVCC_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    BL_PERSIST(p.v, p.pow2, bl_grad_kernel, p.warp_ctas(), st, (const float2*)pts_xy, meta, batch, p.g, p.k, use_bg,
                exact_cull, inv_batch, grad_loss, at<float>(workspace, p.L.amax), at<float>(workspace, p.L.rz),
                at<float>(workspace, p.L.pbg), at<float>(workspace, p.L.wsel), at<float>(workspace, p.L.gpart),
                grad_density, 0, Xchg{}, at<unsigned int>(workspace, p.L.gtick), (int)p.grid.y, at<unsigned int>(workspace, p.L.queue) + 4);
    (void)multi_chunk;  // multi-chunk images are finished inside bl_grad_kernel (last arrival per pixel tile)
    return (int)cudaGetLastError();
}

// ------------------------------------------------------------------- point-chunk sharding: launch sequences
namespace {

struct ShardCtx {
    const dgvcc_bl_shard* sh;
    const dgvcc_bl_push* slices;  // device: DENS and OUT slices
    const unsigned int* aux;      // device: zmask[C] | gmask[C] | img_mask[B] | owner_mask[B]
    char* const* peers;           // device array [world]
    void* ws;
    const dgvcc_bl_layout* L;
    cudaStream_t st;
    int total_chunks, batch;

    const unsigned int* zmask() const { return aux; }
    const unsigned int* gmask() const { return aux + total_chunks; }
    const unsigned int* img_mask() const { return aux + 2 * total_chunks; }
    const unsigned int* owner_mask() const { return aux + 2 * total_chunks + batch; }

    // Xchg of a kernel that produces phase `ph` (mask: per chunk / image destinations; region: exchanged array) and / or
    // waits for `w1`, `w2` first (-1: none).  With separate wait kernels (sh->fuse_waits == 0) the wait part stays empty.
    Xchg make(int ph, const unsigned int* mask, int64_t region, int64_t region2, int w1, int w2) const {
        Xchg x{};
        x.flags = at<unsigned int>(ws, L->flags);
        x.err = at<int>(ws, L->err);
        x.world = sh->world; x.rank = sh->rank; x.epoch = sh->epoch;
        if (ph >= 0) {
            x.peers = peers; x.mask = mask; x.ticket = at<unsigned int>(ws, L->push_ticket);
            x.flags_off = L->flags; x.region_off = region; x.region_off2 = region2;
            x.phase = ph; x.signal_mask = sh->signal_mask[ph];
        }
        if (sh->fuse_waits) {
            if (w1 >= 0) { x.wait_phase = w1; x.wait_mask = sh->wait_mask[w1]; }
            if (w2 >= 0) { x.wait_phase2 = w2; x.wait_mask2 = sh->wait_mask[w2]; }
        }
        return x;
    }
};

// Phase DENS / OUT: copy this rank's slices (sources relative to src_base, destinations relative to the peers' workspaces
// or to dst_override) and, for DENS, raise the flags.
int shard_push(const ShardCtx& c, int ph, const void* src_base, void* dst_override = nullptr, int wait_ph = -1) {
    const int first = c.sh->push_first[ph], n = c.sh->push_first[ph + 1] - first;
    if (!dst_override) {
        if (n <= 0) return DGVCC_OK;
        bl_push_kernel<<<n, PUSH_THREADS, 0, c.st>>>(c.slices + first, n, (const char*)src_base, c.peers, c.L->flags, ph,
                                                     c.sh->rank, c.sh->world, c.sh->signal_mask[ph], c.sh->epoch,
                                                     at<unsigned int>(c.ws, c.L->push_ticket) + 1);  // own counter: side stream
    } else {
        const Xchg x = c.make(-1, nullptr, 0, 0, wait_ph, -1);
        if (n <= 0 && !x.wait_mask) return DGVCC_OK;
        bl_copy_kernel<<<n > 0 ? n : 1, PUSH_THREADS, 0, c.st>>>(c.slices + first, n, (const char*)src_base, (char*)dst_override, x);
    }
    return (int)cudaGetLastError();
}

// Separate wait kernel (sh->fuse_waits == 0: several ranks inside one process / on one GPU, where a whole grid of
// spinning CTAs could keep a co-resident "peer" from ever running).
int shard_wait(const ShardCtx& c, int ph) {
    if (c.sh->fuse_waits || !c.sh->wait_mask[ph]) return DGVCC_OK;
    bl_wait_kernel<<<1, 32, 0, c.st>>>(at<unsigned int>(c.ws, c.L->flags), ph, c.sh->world, c.sh->wait_mask[ph],
                                       c.sh->epoch, XCHG_TIMEOUT_NS, at<int>(c.ws, c.L->err));
    return (int)cudaGetLastError();
}

// The library's side stream and its two events, one set per device: created on first use, handed out once all three exist.
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
SideStream* side_stream() {
    static SideStream side[64];
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return nullptr;
    SideStream& s = side[d];
    if (!s.stream && cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) s.stream = nullptr;
    if (s.stream && !s.fork && cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess) s.fork = nullptr;
    if (s.fork && !s.join && cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess) s.join = nullptr;
    return s.join ? &s : nullptr;
}

// Phase DENS.  The density copy (owner -> sweeping ranks) is needed only by bl_counts, four kernels into the step: it runs
// on the side stream between two events, so it costs the step nothing; *side = nullptr: there is none, it ran on c.st.
int push_density(const ShardCtx& c, const float* density_local, SideStream** side) {
    SideStream* s = *side = c.sh->push_first[DGVCC_BL_PH_DENS + 1] > c.sh->push_first[DGVCC_BL_PH_DENS] ? side_stream() : nullptr;
    if (!s) return shard_push(c, DGVCC_BL_PH_DENS, density_local);
    DGVCC_RETURN_IF_CUDA(cudaEventRecord(s->fork, c.st));
    DGVCC_RETURN_IF_CUDA(cudaStreamWaitEvent(s->stream, s->fork, 0));
    ShardCtx cs = c;
    cs.st = s->stream;
    if (int rc = shard_push(cs, DGVCC_BL_PH_DENS, density_local)) return rc;
    DGVCC_RETURN_IF_CUDA(cudaEventRecord(s->join, s->stream));
    return DGVCC_OK;
}

// Phase OUT, after the GRAD wait: the finished gradients of this rank's own images, gathered into the caller's tensor.
int gather_grad(const ShardCtx& c, float* grad_local) {
    if (int rc = shard_wait(c, DGVCC_BL_PH_GRAD)) return rc;
    if (c.sh->push_first[DGVCC_BL_PH_OUT + 1] > c.sh->push_first[DGVCC_BL_PH_OUT] && !grad_local) return DGVCC_ERR_ARG;
    return shard_push(c, DGVCC_BL_PH_OUT, c.ws, grad_local ? (void*)grad_local : c.ws, DGVCC_BL_PH_GRAD);
}

bool shard_args_ok(const dgvcc_bl_shard* sh, const dgvcc_bl_push* slices, const void* aux, void* const* peers) {
    if (!sh || !peers || !aux) return false;
    for (int ph = 0; ph < DGVCC_BL_PHASES; ++ph)
        if (sh->push_first[ph + 1] < sh->push_first[ph]) return false;
    return sh->push_first[DGVCC_BL_PHASES] == 0 || slices != nullptr;
}

}  // namespace

// CUDA loads kernels lazily, and loading one can wait for the kernels already running in the context: a rank's wait
// kernel spinning on a flag while the kernel that would raise it is still being loaded is a deadlock when several
// ranks share one context (LocalComm), and a stall of the first step otherwise.  Called once per communicator.
extern "C" int dgvcc_bl_shard_preload(void) {
    cudaFuncAttributes a;
#define BL_PRELOAD(K) DGVCC_RETURN_IF_CUDA(cudaFuncGetAttributes(&a, K))
#define BL_PRELOAD_RC(R_, C_)                     \
    BL_PRELOAD((bl_z_kernel<R_, C_, true>));      \
    BL_PRELOAD((bl_z_kernel<R_, C_, false>));     \
    BL_PRELOAD((bl_counts_kernel<R_, C_, true>)); \
    BL_PRELOAD((bl_counts_kernel<R_, C_, false>));\
    BL_PRELOAD((bl_grad_kernel<R_, C_, true>));   \
    BL_PRELOAD((bl_grad_kernel<R_, C_, false>))
    BL_PRELOAD_RC(8, 2);
    BL_PRELOAD_RC(8, 1);
    BL_PRELOAD_RC(4, 1);
    BL_PRELOAD_RC(2, 1);
    BL_PRELOAD(bl_reduce_counts_kernel);
    BL_PRELOAD(bl_select_kernel);
    BL_PRELOAD(bl_grad_reduce_kernel);
    BL_PRELOAD(bl_push_kernel);
    BL_PRELOAD(bl_copy_kernel);
    BL_PRELOAD(bl_wait_kernel);
    BL_PRELOAD(bl_signal_kernel);
    BL_PRELOAD(bl_loss_finish_kernel);
    BL_PRELOAD(bl_grid_build_kernel);
    BL_PRELOAD((bl_gridmin_kernel<2, 1>));
    BL_PRELOAD(bl_finish_z_kernel);
    BL_PRELOAD(bl_band_combine_kernel);
#undef BL_PRELOAD_RC
#undef BL_PRELOAD
    return DGVCC_OK;
}

extern "C" int dgvcc_bl_shard_workspace_layout(int64_t total_rows, int total_chunks, int batch, int hp, int wp, int world,
                                               dgvcc_bl_layout* out) {
    if (world < 1) return DGVCC_ERR_ARG;
    return layout(total_rows, total_chunks, batch, hp, wp, out, world);
}

extern "C" int dgvcc_bl_shard_forward(const float* pts_xy, const float* targets, const int32_t* meta,
                                      const float* st_sizes, const float* density_local, int batch, int hp, int wp,
                                      int64_t total_rows, int total_chunks, int multi_chunk, float stride, float sigma,
                                      float bg_ratio, int use_bg, int exact_cull, float inv_batch,
                                      const dgvcc_bl_shard* shard, const dgvcc_bl_push* slices, const uint32_t* aux,
                                      void* const* peers, void* workspace, size_t workspace_bytes, float* loss_out,
                                      int defer_loss, void* stream, void** events) {
    DGVCC_DEVICE_GUARD(stream);
    if (!shard_args_ok(shard, slices, aux, peers)) return DGVCC_ERR_ARG;
    Plan p;
    int rc = make_plan(meta, st_sizes, workspace, workspace_bytes, batch, hp, wp, total_rows, total_chunks, stride, sigma,
                       &p, shard);
    if (rc) return rc;
    if (!loss_out || !pts_xy || !targets) return DGVCC_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const ShardCtx c{shard, slices, aux, (char* const*)peers, workspace, &p.L, st, total_chunks, batch};
    const float2* pts = (const float2*)pts_xy;
    const bool sweeps = p.grid.y > 0;
    const int n_img = p.sh.img_hi - p.sh.img_lo;
    const int M = hp * wp;
    const dim3 pix_grid(ceil_div(M, 256), n_img > 0 ? n_img : 1);
    mark(events, 0, st);
    // density of the images this rank owns -> every rank that sweeps them (needed from bl_counts on)
    SideStream* side;
    if ((rc = push_density(c, density_local, &side))) return rc;
    mark(events, 1, st);
    // per-pixel minima of the images this rank touches, from ALL their points (replicated on every rank): no exchange
    (void)multi_chunk;
    float* min_img = at<float>(workspace, p.L.pbg);  // the region is free until bl_finish_z_kernel fills it
    if (sweeps && (rc = launch_gridmin(p, pts, meta, batch, hp, wp, p.sh.img_lo, n_img, workspace, min_img, st))) return rc;
    mark(events, 2, st);
    {
        const Xchg x = c.make(DGVCC_BL_PH_Z, c.zmask(), p.L.zpart, 0, -1, -1);
        if (sweeps) {
            BL_PERSIST(p.v, p.pow2, bl_z_kernel, p.warp_ctas(), st, pts, meta, st_sizes, batch, p.g, p.k, bg_ratio, use_bg, exact_cull,
                        at<float>(workspace, p.L.zpart), at<float>(workspace, p.L.amax),
                        at<float>(workspace, p.L.ebg), at<unsigned int>(workspace, p.L.ticket), p.sh, (const float*)min_img, x,
                        at<float>(workspace, p.L.rz), at<float>(workspace, p.L.pbg), at<unsigned int>(workspace, p.L.ztick), 0, (int)p.grid.y, at<unsigned int>(workspace, p.L.queue) + 0);
        } else {
            bl_signal_kernel<<<1, 32, 0, st>>>(x);
        }
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    }
    mark(events, 3, st);
    if (side) DGVCC_RETURN_IF_CUDA(cudaStreamWaitEvent(st, side->join, 0));  // this rank's own copies are in place
    if ((rc = shard_wait(c, DGVCC_BL_PH_Z))) return rc;
    if ((rc = shard_wait(c, DGVCC_BL_PH_DENS))) return rc;
    bl_finish_z_kernel<<<pix_grid, 256, 0, st>>>(meta, batch, M, at<float>(workspace, p.L.zpart), at<float>(workspace, p.L.ebg),
                                                 at<float>(workspace, p.L.rz), at<float>(workspace, p.L.pbg), p.sh.img_lo,
                                                 c.make(-1, nullptr, 0, 0, DGVCC_BL_PH_Z, DGVCC_BL_PH_DENS), n_img);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    mark(events, 4, st);
    if (sweeps) {
        BL_PERSIST(p.v, p.pow2, bl_counts_kernel, (int)(p.grid.x * p.grid.y), st, pts, meta, at<float>(workspace, p.L.dens), batch, p.g, p.k,
                    use_bg, exact_cull, at<float>(workspace, p.L.amax), at<float>(workspace, p.L.rz),
                    at<float>(workspace, p.L.pbg), total_rows, at<float>(workspace, p.L.cpart), -1, Xchg{}, (int)p.grid.y, at<unsigned int>(workspace, p.L.queue) + 2);
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    }
    mark(events, 5, st);
    // fixed-order sums of the tile partials of this rank's rows, delivered to the image's other ranks as they are written
    // (only the rows of the images this rank touches can be its own: the grid covers that window, not the batch)
    const int64_t row_lo = shard->row_lo, row_hi = shard->row_hi > shard->row_lo ? shard->row_hi : shard->row_lo + 1;
    bl_reduce_counts_kernel<<<(unsigned)((row_hi - row_lo + 255) / 256), 256, 0, st>>>(
        at<float>(workspace, p.L.cpart), p.L.tiles, total_rows, meta, targets, batch, at<float>(workspace, p.L.counts),
        at<float>(workspace, p.L.residual), p.sh, c.make(DGVCC_BL_PH_CNT, c.img_mask(), p.L.counts, p.L.residual, -1, -1), row_lo);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    mark(events, 6, st);
    if ((rc = shard_wait(c, DGVCC_BL_PH_CNT))) return rc;
    // top-k cut and per-image loss of every image this rank touches; the rank with an image's first chunk tells everybody
    bl_select_kernel<<<n_img > 0 ? n_img : 1, SELECT_THREADS, 0, st>>>(
        meta, targets, batch, inv_batch, at<float>(workspace, p.L.counts), at<float>(workspace, p.L.residual),
        at<float>(workspace, p.L.wsel), at<float>(workspace, p.L.loss_img), loss_out, at<unsigned int>(workspace, p.L.ticket),
        p.sh.img_lo, 0, p.sh, c.make(DGVCC_BL_PH_LOSS, nullptr, p.L.loss_img, 0, DGVCC_BL_PH_CNT, -1), n_img);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    mark(events, 7, st);
    // the images' losses from all ranks, summed in image order -- a barrier over the whole group, which the backward
    // pass does not need: with defer_loss the same two launches close dgvcc_bl_shard_backward instead
    if (!defer_loss) {
        if ((rc = shard_wait(c, DGVCC_BL_PH_LOSS))) return rc;
        bl_loss_finish_kernel<<<1, 64, 0, st>>>(at<float>(workspace, p.L.loss_img), batch, inv_batch, loss_out,
                                                c.make(-1, nullptr, 0, 0, DGVCC_BL_PH_LOSS, -1));
    }
    mark(events, 8, st);
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_bl_shard_backward(const float* pts_xy, const int32_t* meta, int batch, int hp, int wp,
                                       int64_t total_rows, int total_chunks, float stride, float sigma, int use_bg,
                                       int exact_cull, float inv_batch, const float* grad_loss,
                                       const dgvcc_bl_shard* shard, const dgvcc_bl_push* slices, const uint32_t* aux,
                                       void* const* peers, void* workspace, size_t workspace_bytes, float* grad_local,
                                       float* deferred_loss_out, void* stream, void** events) {
    DGVCC_DEVICE_GUARD(stream);
    if (!shard_args_ok(shard, slices, aux, peers)) return DGVCC_ERR_ARG;
    Plan p;
    int rc = make_plan(meta, grad_loss, workspace, workspace_bytes, batch, hp, wp, total_rows, total_chunks, stride, sigma,
                       &p, shard);
    if (rc) return rc;
    if (!pts_xy) return DGVCC_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const ShardCtx c{shard, slices, aux, (char* const*)peers, workspace, &p.L, st, total_chunks, batch};
    const int M = hp * wp;
    const int n_img = p.sh.img_hi - p.sh.img_lo;
    mark(events, 0, st);
    {   // raw per-chunk gradient sums of every image, written where the rank with the image's first chunk will add them
        const Xchg x = c.make(DGVCC_BL_PH_GPART, c.gmask(), p.L.gpart, 0, -1, -1);
        if (p.grid.y > 0) {
            BL_PERSIST(p.v, p.pow2, bl_grad_kernel, p.warp_ctas(), st, (const float2*)pts_xy, meta, batch, p.g, p.k, use_bg, exact_cull,
                        inv_batch, grad_loss, at<float>(workspace, p.L.amax), at<float>(workspace, p.L.rz),
                        at<float>(workspace, p.L.pbg), at<float>(workspace, p.L.wsel), at<float>(workspace, p.L.gpart),
                        at<float>(workspace, p.L.gfinal), 1, x, at<unsigned int>(workspace, p.L.gtick), (int)p.grid.y, at<unsigned int>(workspace, p.L.queue) + 4);
        } else {
            bl_signal_kernel<<<1, 32, 0, st>>>(x);
        }
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    }
    mark(events, 1, st);
    if ((rc = shard_wait(c, DGVCC_BL_PH_GPART))) return rc;
    // chunk sums added in chunk order, per-pixel factors applied, the result written at the image's owner
    bl_grad_reduce_kernel<<<dim3(ceil_div(M, 256), n_img > 0 ? n_img : 1), 256, 0, st>>>(
        meta, batch, M, use_bg, inv_batch, grad_loss, at<float>(workspace, p.L.gpart), at<float>(workspace, p.L.rz),
        at<float>(workspace, p.L.pbg), at<float>(workspace, p.L.wsel), at<float>(workspace, p.L.gfinal), p.sh,
        c.make(DGVCC_BL_PH_GRAD, c.owner_mask(), p.L.gfinal, 0, DGVCC_BL_PH_GPART, -1), n_img, 0, M, 0);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    mark(events, 2, st);
    rc = gather_grad(c, grad_local);
    mark(events, 3, st);
    if (rc == DGVCC_OK && deferred_loss_out) {  // the loss of a forward that ran with defer_loss
        if ((rc = shard_wait(c, DGVCC_BL_PH_LOSS))) return rc;
        bl_loss_finish_kernel<<<1, 64, 0, st>>>(at<float>(workspace, p.L.loss_img), batch, inv_batch, deferred_loss_out,
                                                c.make(-1, nullptr, 0, 0, DGVCC_BL_PH_LOSS, -1));
        rc = (int)cudaGetLastError();
    }
    mark(events, 4, st);
    return rc;
}

// ------------------------------------------------------------------- row-band sharding: launch sequences
namespace {

// Rows of pixel tiles (R grid rows each) [lo, hi) of rank q's band: as equal as they come, as BandPlan cuts them.
void band_rows(int hp, int R, int world, int q, int* lo, int* hi) {
    const int n_tr = ceil_div(hp, R);
    *lo = (int)((long long)n_tr * q / world);
    *hi = (int)((long long)n_tr * (q + 1) / world);
}

// Plan of a rank that sweeps the grid rows [band_lo, band_hi) of every image over all chunks.
int make_band_plan(const void* a, const void* ws, size_t ws_bytes, int batch, int hp, int wp, int64_t total_rows,
                   int total_chunks, float stride, float sigma, const dgvcc_bl_shard* sh, Plan* p) {
    if (!sh || sh->world < 1 || sh->world > 32 || sh->rank < 0 || sh->rank >= sh->world) return DGVCC_ERR_ARG;
    if (int rc = plan_common(a, ws, ws_bytes, batch, hp, wp, total_rows, total_chunks, stride, sigma, sh->world, p)) return rc;
    const int R = p->v.rows;
    if (sh->band_lo < 0 || sh->band_hi < sh->band_lo || sh->band_hi > hp || sh->band_lo % R != 0 ||
        (sh->band_hi % R != 0 && sh->band_hi != hp))
        return DGVCC_ERR_ARG;   // bands are whole rows of pixel tiles
    int lo, hi;
    band_rows(hp, R, sh->world, sh->rank, &lo, &hi);   // from (hp, R, world) alone: every rank can derive every other rank's
    if (sh->band_lo != (lo * R < hp ? lo * R : hp) || sh->band_hi != (hi * R < hp ? hi * R : hp)) return DGVCC_ERR_ARG;
    p->g.task_first = (sh->band_lo / R) * p->g.col_blocks;
    p->g.tiles = ceil_div(sh->band_hi, R) * p->g.col_blocks;
    p->grid = dim3(ceil_div(p->g.tiles - p->g.task_first, WARPS_PER_CTA), total_chunks);
    return DGVCC_OK;
}

}  // namespace

extern "C" int dgvcc_bl_band_forward(const float* pts_xy, const float* targets, const int32_t* meta, const float* st_sizes,
                                     const float* density_local, int batch, int hp, int wp, int64_t total_rows,
                                     int total_chunks, float stride, float sigma, float bg_ratio, int use_bg, int exact_cull,
                                     float inv_batch, const dgvcc_bl_shard* shard, const dgvcc_bl_push* slices,
                                     const uint32_t* owner_mask, void* const* peers, void* workspace, size_t workspace_bytes,
                                     float* loss_out, void* stream, void** events) {
    DGVCC_DEVICE_GUARD(stream);
    if (!shard_args_ok(shard, slices, owner_mask, peers)) return DGVCC_ERR_ARG;
    Plan p;
    int rc = make_band_plan(meta, workspace, workspace_bytes, batch, hp, wp, total_rows, total_chunks, stride, sigma, shard, &p);
    if (rc) return rc;
    if (!loss_out || !pts_xy || !targets || !st_sizes) return DGVCC_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const ShardCtx c{shard, slices, owner_mask, (char* const*)peers, workspace, &p.L, st, total_chunks, batch};
    const float2* pts = (const float2*)pts_xy;
    const bool sweeps = p.grid.x > 0 && p.grid.y > 0;
    mark(events, 0, st);
    // density rows of the images this rank owns -> the ranks whose bands they fall into (needed from bl_counts on)
    SideStream* side;
    if ((rc = push_density(c, density_local, &side))) return rc;
    mark(events, 1, st);
    float* min_img = at<float>(workspace, p.L.gpart);  // free until the backward pass
    if (sweeps) {
        if ((rc = launch_gridmin(p, pts, meta, batch, hp, wp, 0, batch, workspace, min_img, st, shard->band_lo, shard->band_hi)))
            return rc;
        mark(events, 2, st);
        BL_PERSIST(p.v, p.pow2, bl_z_kernel, p.warp_ctas(), st, pts, meta, st_sizes, batch, p.g, p.k, bg_ratio, use_bg, exact_cull,
                    at<float>(workspace, p.L.zpart), at<float>(workspace, p.L.amax), at<float>(workspace, p.L.ebg),
                    at<unsigned int>(workspace, p.L.ticket), p.sh, (const float*)min_img, Xchg{}, at<float>(workspace, p.L.rz),
                    at<float>(workspace, p.L.pbg), at<unsigned int>(workspace, p.L.ztick), 1, (int)p.grid.y, at<unsigned int>(workspace, p.L.queue) + 0);
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    } else {
        mark(events, 2, st);
    }
    mark(events, 3, st);
    if (side) DGVCC_RETURN_IF_CUDA(cudaStreamWaitEvent(st, side->join, 0));
    if ((rc = shard_wait(c, DGVCC_BL_PH_DENS))) return rc;
    // expected counts: every CTA stores its partial row into the count-share table of EVERY rank as it is produced
    // (rows [rank * share_rows, ...)); the kernel's last CTA raises CNT
    const Xchg cnt = c.make(DGVCC_BL_PH_CNT, nullptr, p.L.cshare, 0, DGVCC_BL_PH_DENS, -1);
    if ((int)p.grid.x > p.L.share_rows) return DGVCC_ERR_ARG;
    if (sweeps) {
        BL_PERSIST(p.v, p.pow2, bl_counts_kernel, (int)(p.grid.x * p.grid.y), st, pts, meta, at<float>(workspace, p.L.dens), batch, p.g, p.k,
                    use_bg, exact_cull, at<float>(workspace, p.L.amax), at<float>(workspace, p.L.rz),
                    at<float>(workspace, p.L.pbg), total_rows, (float*)nullptr, shard->rank * p.L.share_rows, cnt, (int)p.grid.y, at<unsigned int>(workspace, p.L.queue) + 2);
    } else {
        bl_signal_kernel<<<1, 32, 0, st>>>(cnt);
    }
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    mark(events, 4, st);
    if ((rc = shard_wait(c, DGVCC_BL_PH_CNT))) return rc;
    // every rank adds all partial rows in (rank, CTA) order -- the order of the pixel tiles, as on one GPU
    BandRows br{};
    for (int q = 0; q < shard->world; ++q) {  // the bands of all ranks follow from (hp, R, world) alone
        int lo, hi;
        band_rows(hp, p.v.rows, shard->world, q, &lo, &hi);
        br.n[q] = ceil_div((hi - lo) * p.g.col_blocks, WARPS_PER_CTA);
    }
    const unsigned row_blocks = (unsigned)((total_rows + 255) / 256);
    bl_band_combine_kernel<<<row_blocks, 256, 0, st>>>(at<float>(workspace, p.L.cshare), shard->world, p.L.share_rows, br,
                                                       total_rows, meta, targets, batch, at<float>(workspace, p.L.counts),
                                                       at<float>(workspace, p.L.residual),
                                                       c.make(-1, nullptr, 0, 0, DGVCC_BL_PH_CNT, -1));
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    mark(events, 5, st);
    // top-k cut and loss of every image, on every rank (the same bits everywhere): no exchange
    bl_select_kernel<<<batch, SELECT_THREADS, 0, st>>>(
        meta, targets, batch, inv_batch, at<float>(workspace, p.L.counts), at<float>(workspace, p.L.residual),
        at<float>(workspace, p.L.wsel), at<float>(workspace, p.L.loss_img), loss_out, at<unsigned int>(workspace, p.L.ticket),
        0, 1, no_shard(), Xchg{}, batch);
    mark(events, 6, st);
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_bl_band_backward(const float* pts_xy, const int32_t* meta, int batch, int hp, int wp, int64_t total_rows,
                                      int total_chunks, float stride, float sigma, int use_bg, int exact_cull, float inv_batch,
                                      const float* grad_loss, const dgvcc_bl_shard* shard, const dgvcc_bl_push* slices,
                                      const uint32_t* owner_mask, void* const* peers, void* workspace, size_t workspace_bytes,
                                      float* grad_local, void* stream, void** events) {
    DGVCC_DEVICE_GUARD(stream);
    if (!shard_args_ok(shard, slices, owner_mask, peers)) return DGVCC_ERR_ARG;
    Plan p;
    int rc = make_band_plan(meta, workspace, workspace_bytes, batch, hp, wp, total_rows, total_chunks, stride, sigma, shard, &p);
    if (rc) return rc;
    if (!pts_xy || !grad_loss) return DGVCC_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const ShardCtx c{shard, slices, owner_mask, (char* const*)peers, workspace, &p.L, st, total_chunks, batch};
    const bool sweeps = p.grid.x > 0 && p.grid.y > 0;
    mark(events, 0, st);
    // gradient of the band's pixels, finished inside the sweep (last arrival per pixel tile) and written at the image's owner
    const Xchg out = c.make(DGVCC_BL_PH_GRAD, owner_mask, p.L.gfinal, 0, -1, -1);
    if (sweeps) {
        BL_PERSIST(p.v, p.pow2, bl_grad_kernel, p.warp_ctas(), st, (const float2*)pts_xy, meta, batch, p.g, p.k, use_bg, exact_cull,
                    inv_batch, grad_loss, at<float>(workspace, p.L.amax), at<float>(workspace, p.L.rz),
                    at<float>(workspace, p.L.pbg), at<float>(workspace, p.L.wsel), at<float>(workspace, p.L.gpart),
                    at<float>(workspace, p.L.gfinal), 0, out, at<unsigned int>(workspace, p.L.gtick), (int)p.grid.y, at<unsigned int>(workspace, p.L.queue) + 4);
    } else {
        bl_signal_kernel<<<1, 32, 0, st>>>(out);
    }
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    mark(events, 1, st);
    rc = gather_grad(c, grad_local);
    mark(events, 2, st);
    return rc;
}

// ------------------------------------------------------------------- peer memory (CUDA IPC) for the sharded path
extern "C" int dgvcc_peer_alloc(size_t bytes, void** ptr) {
    if (!ptr || bytes == 0) return DGVCC_ERR_ARG;
    DGVCC_RETURN_IF_CUDA(cudaMalloc(ptr, bytes));
    DGVCC_RETURN_IF_CUDA(cudaMemset(*ptr, 0, bytes));
    return (int)cudaDeviceSynchronize();
}
extern "C" int dgvcc_peer_free(void* ptr) { return ptr ? (int)cudaFree(ptr) : DGVCC_OK; }
extern "C" int dgvcc_peer_export(void* ptr, unsigned char* handle64) {
    if (!ptr || !handle64) return DGVCC_ERR_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    return (int)cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle64), ptr);
}
extern "C" int dgvcc_peer_open(const unsigned char* handle64, void** ptr) {
    if (!ptr || !handle64) return DGVCC_ERR_ARG;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    return (int)cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
}
extern "C" int dgvcc_peer_close(void* ptr) { return ptr ? (int)cudaIpcCloseMemHandle(ptr) : DGVCC_OK; }

extern "C" int dgvcc_bl_posterior(const float* pts_xy, const int32_t* meta, const float* st_sizes, int batch,
                                  int hp, int wp, int64_t total_rows, int total_chunks, int multi_chunk,
                                  float stride, float sigma, float bg_ratio, int use_bg, void* workspace,
                                  size_t workspace_bytes, float* prob_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    Plan p;
    int rc = make_plan(meta, st_sizes, workspace, workspace_bytes, batch, hp, wp, total_rows, total_chunks, stride,
                       sigma, &p);
    if (rc) return rc;
    if (!prob_out || !pts_xy) return DGVCC_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = launch_z(p, pts_xy, meta, st_sizes, batch, multi_chunk, bg_ratio, use_bg, /*exact_cull=*/0, workspace, st))) return rc;
    const int M = hp * wp;
    bl_finish_z_kernel<<<dim3(ceil_div(M, 256), batch), 256, 0, st>>>(
        meta, batch, M, at<float>(workspace, p.L.zpart), at<float>(workspace, p.L.ebg), at<float>(workspace, p.L.rz),
        at<float>(workspace, p.L.pbg), 0, Xchg{}, batch);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    BL_DISPATCH(p.v, p.pow2, bl_posterior_kernel, p.grid, st, (const float2*)pts_xy, meta, batch, p.g, p.k, use_bg,
                at<float>(workspace, p.L.amax), at<float>(workspace, p.L.rz), at<float>(workspace, p.L.pbg), prob_out);
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_bl_bayloss_forward(const float* prob, const float* targets, const int32_t* meta,
                                        const float* density, int batch, int hp, int wp, int64_t total_rows,
                                        float inv_batch, void* workspace, size_t workspace_bytes,
                                        float* loss_out, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!prob || !targets || !meta || !density || !workspace || !loss_out) return DGVCC_ERR_ARG;
    dgvcc_bl_layout L;
    int rc;
    if ((rc = layout(total_rows, batch, batch, hp, wp, &L))) return rc;
    if (workspace_bytes < (size_t)L.total) return DGVCC_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int M = hp * wp;
    bl_prob_counts_kernel<<<(unsigned)((total_rows + 7) / 8), 256, 0, st>>>(prob, density, meta, batch, M, total_rows,
                                                                            at<float>(workspace, L.cpart),
                                                                            at<unsigned int>(workspace, L.ticket));
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    return launch_select(L, targets, meta, batch, total_rows, inv_batch, /*tiles=*/1, workspace, loss_out, st);
}

extern "C" int dgvcc_bl_bayloss_backward(const float* prob, const int32_t* meta, int batch, int hp, int wp,
                                         int64_t total_rows, float inv_batch, const float* grad_loss,
                                         const void* workspace, size_t workspace_bytes, float* grad_density,
                                         void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (!prob || !meta || !grad_loss || !workspace || !grad_density) return DGVCC_ERR_ARG;
    dgvcc_bl_layout L;
    int rc;
    if ((rc = layout(total_rows, batch, batch, hp, wp, &L))) return rc;
    if (workspace_bytes < (size_t)L.total) return DGVCC_ERR_WORKSPACE;
    const int M = hp * wp;
    bl_prob_grad_kernel<<<dim3(ceil_div(M, 256), batch), 256, 0, (cudaStream_t)stream>>>(
        prob, meta, batch, M, inv_batch, grad_loss, at<float>(workspace, L.wsel), grad_density);
    return (int)cudaGetLastError();
}
