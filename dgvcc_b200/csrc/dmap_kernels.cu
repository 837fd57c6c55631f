// Geometry-adaptive density-map generation for sm_100a.
//
// Replaces utils/dmap_gen.py:14-81 of the reference (scipy KDTree k=4 query + one full-image
// scipy.ndimage.gaussian_filter per head).  A whole list of images goes through one set of launches
// (dgvcc_dmap_batch_plan lays out the work; `meta` is its per-image table):
//   dmap_knn_batch_kernel : brute-force tiled 4-nearest search, exact in fp64 (self included, like
//   + prep / merge          KDTree.query(points, k=4)) behind an exact fp32 filter, candidates in slices across CTAs,
//                           two phases (slice 0 bounds the others); sigma = 0.1*(d1+d2+d3)   dmap_gen.py:34-48
//                           (dmap_knn_kernel + dmap_knn_merge_kernel: the single-image form behind knn_sigma())
//   dmap_prepare_kernel   : per head: truncated pixel index, in-bounds test, kernel radius
//   / _fixed_ variants      int(truncate*sigma+0.5), the normaliser of scipy's 1-D Gaussian kernel summed in numpy's
//                           pairwise order, bounding box, weight table of narrow stamps, tile occupancy bits
//                                                                                           dmap_gen.py:41-49
//   dmap_coarse_kernel    : ordered two-level culling: per 256x256 coarse tile the list of heads whose stamp touches
//   dmap_tile_setup_kernel  it, IN INDEX ORDER (count pass + write pass); one descriptor per 32x32 fine tile
//   dmap_splat_kernel     : one CTA per 32x32 output tile gathers, from its coarse list, the heads whose stamp
//                           overlaps it, in index order, and accumulates fl32(f64(fl32(w[dy])) * w[dx]) per pixel
//                           in fp32 -- the closed form of gaussian_filter on a one-hot image (SURVEY.md 8c).
//                           Every output pixel is written exactly once (zero fill fused), coalesced.
// All fp64 arithmetic uses explicit _rn intrinsics (no FMA contraction): scipy's wheels are baseline
// x86-64 without FMA, and the neighbour indices must match bit for bit.
#include <math.h>

#include "common.cuh"
#include "../../include/dgvcc_b200.h"

namespace dgvcc {
namespace dmap {

constexpr int KNN_THREADS = 256;

// ---------------------------------------------------------------------------------- kNN + sigma
// Each CTA finds, for its 256 query heads, the 4 nearest candidates inside one slice of the head list
// (grid.y slices, so that small and large N both fill the chip); dmap_knn_merge_kernel then merges the
// per-slice lists.  Order is (squared distance, index) everywhere, so ties keep the lower index.
__device__ __forceinline__ void knn_insert(double (&best)[4], int (&bidx)[4], double d2, int j) {
    best[3] = d2; bidx[3] = j;
#pragma unroll
    for (int k = 3; k > 0; --k) {
        if (best[k] < best[k - 1] || (best[k] == best[k - 1] && bidx[k] < bidx[k - 1])) {
            const double tb = best[k]; best[k] = best[k - 1]; best[k - 1] = tb;
            const int ti = bidx[k]; bidx[k] = bidx[k - 1]; bidx[k - 1] = ti;
        }
    }
}

__global__ void __launch_bounds__(KNN_THREADS)
dmap_knn_kernel(const double2* __restrict__ pts, int n, int slice_len, double* __restrict__ part_d2,
                int32_t* __restrict__ part_idx) {
    __shared__ double2 cand[KNN_THREADS];
    const int i = blockIdx.x * KNN_THREADS + threadIdx.x;
    const double2 q = pts[min(i, n - 1)];
    double best[4];
    int bidx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { best[k] = INFINITY; bidx[k] = n; }  // scipy: missing neighbour = (inf, N)
    const int j_begin = blockIdx.y * slice_len, j_end = min(n, j_begin + slice_len);
    for (int j0 = j_begin; j0 < j_end; j0 += KNN_THREADS) {
        __syncthreads();
        if (j0 + threadIdx.x < j_end) cand[threadIdx.x] = pts[j0 + threadIdx.x];
        __syncthreads();
        const int lim = min(KNN_THREADS, j_end - j0);
#pragma unroll 4
        for (int t = 0; t < lim; ++t) {
            const double dx = __dsub_rn(q.x, cand[t].x);
            const double dy = __dsub_rn(q.y, cand[t].y);
            const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
            // candidates arrive in index order, so on ties the earlier (lower) index stays in front
            if (d2 < best[3]) knn_insert(best, bidx, d2, j0 + t);
        }
    }
    if (i >= n) return;
    const size_t o = ((size_t)blockIdx.y * n + i) * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) { part_d2[o + k] = best[k]; part_idx[o + k] = bidx[k]; }
}

__global__ void __launch_bounds__(KNN_THREADS)
dmap_knn_merge_kernel(const double* __restrict__ part_d2, const int32_t* __restrict__ part_idx, int n, int slices,
                      int32_t* __restrict__ nn_idx, double* __restrict__ nn_dist, double* __restrict__ sigma) {
    const int i = blockIdx.x * KNN_THREADS + threadIdx.x;
    if (i >= n) return;
    double best[4];
    int bidx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { best[k] = INFINITY; bidx[k] = n; }
    for (int s = 0; s < slices; ++s) {
        const size_t o = ((size_t)s * n + i) * 4;
        for (int k = 0; k < 4; ++k) {
            const double d2 = part_d2[o + k];
            const int j = part_idx[o + k];
            if (j < n && (d2 < best[3] || (d2 == best[3] && j < bidx[3]))) knn_insert(best, bidx, d2, j);
        }
    }
    double d[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        d[k] = __dsqrt_rn(best[k]);
        nn_idx[4 * i + k] = bidx[k];
        nn_dist[4 * i + k] = d[k];
    }
    // dmap_gen.py:45-48: (d1 + d2 + d3) * 0.1 when there are more than 3 heads, else 15
    sigma[i] = (n > 3) ? __dmul_rn(__dadd_rn(__dadd_rn(d[1], d[2]), d[3]), 0.1) : 15.0;
}

// ---------------------------------------------------------------------------- per-head stamp data
struct Stamp {
    int ix, iy;      // pixel of the one-hot write (dmap_gen.py:42), after numpy's negative-index wrap
    int radius;      // int(truncate * sigma + 0.5); -1 marks a skipped head (dmap_gen.py:41-44)
    int pad_;
    double coef;     // -0.5 / sigma^2
    double norm;     // sum of exp(coef * i^2), i = -radius..radius, in numpy's pairwise order
};

__device__ __forceinline__ double phi(double coef, int i) {
    return exp(__dmul_rn(coef, (double)((long long)i * i)));
}

// Leaf of numpy's pairwise summation (DOUBLE_pairwise_sum, n <= 128) over phi(first), phi(first+1), ...
__device__ __forceinline__ double pairwise_leaf(double coef, int first, int n) {
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = __dadd_rn(res, phi(coef, first + i));
        return res;
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = phi(coef, first + j);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], phi(coef, first + i + j));
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, phi(coef, first + i));
    return res;
}

// numpy's pairwise summation: blocks of <= 128 are leaves, larger ranges split at n/2 rounded down to a
// multiple of 8 and the halves are added.  Explicit stack instead of recursion (depth <= 24 for n < 2^31),
// so the kernel needs no enlarged device stack however large a sparse image's sigma gets.
__device__ double pairwise_phi_sum(double coef, int first, int n) {
    constexpr int DEPTH = 26;
    int s_first[DEPTH], s_n[DEPTH], s_stage[DEPTH];
    double s_left[DEPTH];
    int sp = 0;
    s_first[0] = first; s_n[0] = n; s_stage[0] = 0;
    double ret = 0.0;
    while (sp >= 0) {
        const int cn = s_n[sp];
        int n2 = cn / 2;
        n2 -= n2 % 8;
        if (s_stage[sp] == 0) {
            if (cn <= 128) { ret = pairwise_leaf(coef, s_first[sp], cn); --sp; continue; }
            s_stage[sp] = 1;
            s_first[sp + 1] = s_first[sp]; s_n[sp + 1] = n2; s_stage[sp + 1] = 0;
            ++sp;
        } else if (s_stage[sp] == 1) {
            s_left[sp] = ret;
            s_stage[sp] = 2;
            s_first[sp + 1] = s_first[sp] + n2; s_n[sp + 1] = cn - n2; s_stage[sp + 1] = 0;
            ++sp;
        } else {
            ret = __dadd_rn(s_left[sp], ret);
            --sp;
        }
    }
    return ret;
}

// ---- the same sum, one warp per head -------------------------------------------------------------
// Groups of 8 lanes evaluate one leaf each: lane j of a group owns numpy's accumulator r[j] (elements
// j, j+8, ... of the leaf), the group leader combines them in numpy's order and adds the tail.  The tree above
// the leaves is then combined by lane 0 in numpy's recursion order.  Bit-identical to pairwise_phi_sum.
constexpr int MAX_LEAVES = 256;

struct LeafList {
    int first[MAX_LEAVES];
    int len[MAX_LEAVES];
    double sum[MAX_LEAVES];
};

// DFS enumeration of the leaves of numpy's recursion over [first, first + n); returns their number
// (or -1 when there are more than MAX_LEAVES).  Pure integer work, done redundantly by every lane.
__device__ int enumerate_leaves(int first, int n, LeafList& ll, bool write) {
    constexpr int DEPTH = 26;
    int s_first[DEPTH], s_n[DEPTH], s_stage[DEPTH];
    int sp = 0, count = 0;
    s_first[0] = first; s_n[0] = n; s_stage[0] = 0;
    while (sp >= 0) {
        const int cn = s_n[sp];
        int n2 = cn / 2;
        n2 -= n2 % 8;
        if (s_stage[sp] == 0) {
            if (cn <= 128) {
                if (count >= MAX_LEAVES) return -1;
                if (write) { ll.first[count] = s_first[sp]; ll.len[count] = cn; }
                ++count; --sp;
                continue;
            }
            s_stage[sp] = 1;
            s_first[sp + 1] = s_first[sp]; s_n[sp + 1] = n2; s_stage[sp + 1] = 0;
            ++sp;
        } else if (s_stage[sp] == 1) {
            s_stage[sp] = 2;
            s_first[sp + 1] = s_first[sp] + n2; s_n[sp + 1] = cn - n2; s_stage[sp + 1] = 0;
            ++sp;
        } else {
            --sp;
        }
    }
    return count;
}

// One leaf (n <= 128) by a group of 8 lanes; the result is valid on the group's lane 0.
__device__ __forceinline__ double leaf_by_group(double coef, int first, int n, int sub /*0..7*/, unsigned group_mask) {
    const int group_lane0 = __ffs(group_mask) - 1;  // first lane of this group of 8
    if (n < 8) {  // numpy's plain loop: the lanes evaluate the elements side by side, the leader adds them in order
        const double ev = sub < n ? phi(coef, first + sub) : 0.0;
        double res = 0.0;
        for (int j = 0; j < n; ++j) {
            const double v = __shfl_sync(group_mask, ev, (group_lane0 + j) & 31);
            if (sub == 0) res = __dadd_rn(res, v);
        }
        return res;
    }
    const int body = n - (n % 8);
    double r = phi(coef, first + sub);
    for (int i = 8; i < body; i += 8) r = __dadd_rn(r, phi(coef, first + i + sub));
    // ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7)): a butterfly over the 8 lanes is exactly this tree
    r = __dadd_rn(r, __shfl_xor_sync(group_mask, r, 1));
    r = __dadd_rn(r, __shfl_xor_sync(group_mask, r, 2));
    r = __dadd_rn(r, __shfl_xor_sync(group_mask, r, 4));
    // numpy adds the n % 8 tail elements one by one: the lanes evaluate them side by side (sub-lane j holds tail
    // element j), the leader then adds them in order
    const int tail = n - body;
    const double tv = sub < tail ? phi(coef, first + body + sub) : 0.0;
    for (int j = 0; j < tail; ++j) {
        const double v = __shfl_sync(group_mask, tv, (group_lane0 + j) & 31);
        if (sub == 0) r = __dadd_rn(r, v);
    }
    return r;
}

// Combine the leaf sums in numpy's recursion order (lane 0 only).
__device__ double combine_leaves(int first, int n, const LeafList& ll) {
    constexpr int DEPTH = 26;
    int s_n[DEPTH], s_stage[DEPTH];
    double s_left[DEPTH];
    int sp = 0, next = 0;
    s_n[0] = n; s_stage[0] = 0;
    double ret = 0.0;
    (void)first;
    while (sp >= 0) {
        const int cn = s_n[sp];
        int n2 = cn / 2;
        n2 -= n2 % 8;
        if (s_stage[sp] == 0) {
            if (cn <= 128) { ret = ll.sum[next++]; --sp; continue; }
            s_stage[sp] = 1; s_n[sp + 1] = n2; s_stage[sp + 1] = 0; ++sp;
        } else if (s_stage[sp] == 1) {
            s_left[sp] = ret; s_stage[sp] = 2; s_n[sp + 1] = cn - n2; s_stage[sp + 1] = 0; ++sp;
        } else {
            ret = __dadd_rn(s_left[sp], ret); --sp;
        }
    }
    return ret;
}

// ------------------------------------------------------------------------------ batch bookkeeping
// One launch handles a whole list of images.  The host plan (dgvcc_dmap_batch_plan) writes one row of
// META_COLS int64 per image plus a final row of totals; kernels find the image of a CTA / head by binary
// search over the cumulative columns (L1-resident after the first touch).
enum MetaCol {
    M_PT_OFF = 0,    // first head of the image in the packed head arrays
    M_N = 1,         // heads
    M_H = 2,
    M_W = 3,
    M_OUT_OFF = 4,   // first float of the image in the packed output
    M_FTILE_OFF = 5, // first fine-tile CTA
    M_CTASK_OFF = 6, // first coarse task (coarse tile x head chunk)
    M_CLIST_OFF = 7, // first entry of the image's coarse lists (coarse tiles x n entries)
    M_CTILE_OFF = 8, // first coarse tile (index into ctotal / ccount rows)
    M_KTASK_OFF = 9, // first kNN task (query block x candidate slice)
    M_KPART_OFF = 10,// first entry of the image's kNN partial lists (slices x n x 4)
    M_KQB_OFF = 11,  // first kNN query block (256 heads)
    META_COLS = DGVCC_DMAP_META_COLS
};
static_assert(META_COLS == 12, "header and kernels disagree on the meta row width");

constexpr int FINE_W = 32;        // fine tile: 32 columns (one warp row) x FINE_H rows
constexpr int SPLAT_RPT = 8;      // rows per thread
constexpr int SPLAT_WARPS = 4;
constexpr int SPLAT_THREADS = SPLAT_WARPS * 32;
constexpr int FINE_H = SPLAT_WARPS * SPLAT_RPT;  // 32
constexpr int COARSE_THREADS = 256;
constexpr int COARSE = 256;       // coarse tile side, a multiple of both fine sides
constexpr int CHUNK = 2048;       // heads per coarse task
constexpr int KNN_SLICE = 2048;   // fewest candidates per batched kNN task

// Candidate slices of an image with n heads: at most max_slices equal slices of at least KNN_SLICE candidates.
// Every slice restarts its neighbour list, which costs insertions, so a batch that already fills the chip with
// query blocks uses few slices and a single big image uses many.  Slice 0 is scanned first (phase 0) and gives
// the others (phase 1) their bound.  (Measured on the 64-image set: a short bound-only slice 0 plus long phase-1
// slices is slower -- 1.39 vs 1.26 ms -- than equal halves: the bound of a longer scan is tighter.)
struct KnnSlicing {
    int first_len, rest, rest_len;
    __host__ __device__ int slices() const { return 1 + rest; }
    __host__ __device__ int begin(int s) const { return s == 0 ? 0 : first_len + (s - 1) * rest_len; }
    __host__ __device__ int len(int s) const { return s == 0 ? first_len : rest_len; }
};
__host__ __device__ __forceinline__ KnnSlicing knn_slicing(int n, int max_slices) {
    KnnSlicing k;
    int s = (n + KNN_SLICE - 1) / KNN_SLICE;
    if (s > max_slices) s = max_slices;
    if (s < 1) s = 1;
    const int len = ((n + s - 1) / s + 255) / 256 * 256;
    k.first_len = n < len ? n : len;
    k.rest_len = len;
    k.rest = (n - k.first_len + len - 1) / len;
    return k;
}
constexpr int TAB = 32;           // stamps of radius < TAB read their weights from the per-head table
constexpr int GROUP = 32;         // heads staged together by a fine tile (<= 64: masks are 64-bit)
constexpr int GEN_MAX = 8;        // of which at most this many wide ones (radius >= TAB: weights evaluated per tile)

// last row r < rows with meta[r][col] <= v (cumulative column, meta[0][col] = 0; callers pass the image rows
// plus the row of totals, which is never selected because v < total; images that own nothing are skipped)
__device__ __forceinline__ int find_image(const int64_t* __restrict__ meta, int rows, int col, int64_t v) {
    int lo = 0, hi = rows;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(meta + (size_t)mid * META_COLS + col) <= v) lo = mid; else hi = mid;
    }
    return lo;
}

// ------------------------------------------------------------------------------- batched kNN
// fp32 copies of the heads + the largest |coordinate| of every image (for the error bound of the fp32 filter).
__global__ void __launch_bounds__(256)
dmap_knn_prep_kernel(const double2* __restrict__ pts, const int64_t* __restrict__ meta, int n_images, int total_heads,
                     float2* __restrict__ pts32, int* __restrict__ img_max_bits) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total_heads) return;
    const double2 p = pts[g];
    pts32[g] = make_float2(__double2float_rn(p.x), __double2float_rn(p.y));
    const float m = __double2float_ru(fmax(fabs(p.x), fabs(p.y)));  // non-negative floats order like their bit patterns
    const int img = find_image(meta, n_images + 1, M_PT_OFF, g);
    // one atomic per (warp, image): lanes of the same image reduce among themselves first
    const unsigned peers = __match_any_sync(__activemask(), img);
    const int warp_max = __reduce_max_sync(peers, __float_as_int(m));
    if ((threadIdx.x & 31) == __ffs(peers) - 1 && warp_max > img_max_bits[img]) atomicMax(img_max_bits + img, warp_max);
}

// Upper bound, in fp32, of what the fp32 evaluation of a squared distance can return when the exact fp64 value is
// below `thr`.  With u = 2^-24, M >= every |coordinate| of the image and d2 the exact value, the fp32 result is within
//     E(d2) <= 5.7 u M sqrt(d2) + 4.2 u d2 + 16 u^2 M^2
// of d2 (inputs rounded to fp32: <= u M each; the difference, the two squares and the sum: relative u each); E grows
// with d2, so d2 < thr implies fp32(d2) <= thr + E(thr).  The constants below are more than twice the derived ones and
// every step rounds up.  Candidates above the bound are skipped, all others are evaluated exactly in fp64.
__device__ __forceinline__ float knn_bound32(double thr, float big_m) {
    if (!(thr < 1.0e30) || !(big_m < 1.0e15f)) return INFINITY;  // nothing to filter with / out of the bound's range
    constexpr float U = 5.9604645e-8f;
    const float t = __double2float_ru(thr);
    const float um = __fmul_ru(U, big_m);
    float e = __fmul_ru(__fmul_ru(12.f, um), __fmul_ru(__fsqrt_ru(t), 1.000001f));
    e = __fadd_ru(e, __fmul_ru(__fmul_ru(16.f, U), t));
    e = __fadd_ru(e, __fmul_ru(32.f, __fmul_ru(um, um)));
    return __fadd_ru(t, e);
}

// Task = (image, block of 256 query heads, slice of KNN_SLICE candidates); the merge kernel combines the
// per-slice lists.  Same fp64 arithmetic and (distance, index) order as the single-image kernels above.
// Two things keep the FP64 pipe (the bound of the plain brute-force loop) out of the inner loop:
// * an fp32 filter: the squared distance is first evaluated in fp32 (4 instructions on the FP32 pipe) and compared
//   with knn_bound32 of the current threshold; only candidates that pass are evaluated in fp64, exactly as before,
//   so the result is unchanged bit for bit;
// * two phases: a slice that starts from an empty list inserts all the time, and one inserting lane drags its whole
//   warp through the insertion network.  Phase 0 runs slice 0 of every query block, phase 1 (all other slices)
//   starts each query with the 4th-best distance of its slice 0 as an upper bound: a later candidate at that
//   distance or beyond cannot enter the final list (later slices hold higher indices, which lose ties).
__global__ void __launch_bounds__(KNN_THREADS)
dmap_knn_batch_kernel(const double2* __restrict__ pts, const float2* __restrict__ pts32, const int* __restrict__ img_max_bits,
                      const int64_t* __restrict__ meta, int n_images, int max_slices, int phase,
                      double* __restrict__ part_d2, int32_t* __restrict__ part_idx) {
    __shared__ double2 cand[KNN_THREADS];
    __shared__ float4 cand32[KNN_THREADS / 2];  // fp32 candidates, negated, in pairs: (-x0, -x1, -y0, -y1)
    int img, slice, qb;
    if (phase == 0) {
        img = find_image(meta, n_images + 1, M_KQB_OFF, blockIdx.x);
        slice = 0;
        qb = blockIdx.x - (int)meta[(size_t)img * META_COLS + M_KQB_OFF];
    } else {
        // cumulative count of phase-1 tasks = all tasks - query blocks
        int lo = 0, hi = n_images + 1;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            const int64_t* mm = meta + (size_t)mid * META_COLS;
            if (__ldg(mm + M_KTASK_OFF) - __ldg(mm + M_KQB_OFF) <= (int64_t)blockIdx.x) lo = mid; else hi = mid;
        }
        img = lo;
        const int64_t* mm = meta + (size_t)img * META_COLS;
        const int rest = knn_slicing((int)mm[M_N], max_slices).rest;
        const int local = blockIdx.x - (int)(mm[M_KTASK_OFF] - mm[M_KQB_OFF]);
        slice = 1 + local % rest;
        qb = local / rest;
    }
    const int64_t* m = meta + (size_t)img * META_COLS;
    const int n = (int)m[M_N];
    const double2* p = pts + m[M_PT_OFF];
    const float2* p32 = pts32 + m[M_PT_OFF];
    const float big_m = __int_as_float(img_max_bits[img]);
    const int i = qb * KNN_THREADS + threadIdx.x;
    const double2 q = p[min(i, n - 1)];
    const float2 qf = p32[min(i, n - 1)];
    double best[4];
    int bidx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { best[k] = INFINITY; bidx[k] = n; }
    const double bound = phase == 0 ? INFINITY : part_d2[(size_t)m[M_KPART_OFF] + (size_t)min(i, n - 1) * 4 + 3];
    double thr = bound;  // = min(best[3], bound)
    float thr32 = knn_bound32(thr, big_m);
    const f2 qx2 = pack2(qf.x, qf.x), qy2 = pack2(qf.y, qf.y);
    const KnnSlicing ks = knn_slicing(n, max_slices);
    const int j_begin = ks.begin(slice), j_end = min(n, j_begin + ks.len(slice));
    for (int j0 = j_begin; j0 < j_end; j0 += KNN_THREADS) {
        __syncthreads();
        {
            // candidates past the end of the slice become +inf: their fp32 distance is inf and never passes
            float2 c = make_float2(-INFINITY, -INFINITY);
            if (j0 + threadIdx.x < j_end) {
                cand[threadIdx.x] = p[j0 + threadIdx.x];
                c = p32[j0 + threadIdx.x];
            }
            float* c32 = reinterpret_cast<float*>(cand32) + 4 * (threadIdx.x >> 1) + (threadIdx.x & 1);
            c32[0] = -c.x;
            c32[2] = -c.y;
        }
        __syncthreads();
        const int lim = min(KNN_THREADS, j_end - j0);
        auto exact = [&](int t) {  // the reference's fp64 evaluation, for a candidate the fp32 filter let through
            const double dx = __dsub_rn(q.x, cand[t].x);
            const double dy = __dsub_rn(q.y, cand[t].y);
            const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
            if (d2 < thr) {
                knn_insert(best, bidx, d2, j0 + t);
                thr = fmin(best[3], bound);
                thr32 = knn_bound32(thr, big_m);
            }
        };
        // two candidates per step with Blackwell's packed fp32x2 add / mul / fma (each half an ordinary IEEE op)
#pragma unroll 4
        for (int t = 0; t < lim; t += 2) {
            const ulonglong2 c = *reinterpret_cast<const ulonglong2*>(&cand32[t >> 1]);  // {(-x0,-x1), (-y0,-y1)}
            const f2 fx = add2(qx2, c.x), fy = add2(qy2, c.y);
            float a0, a1;
            unpack2(fma2(fx, fx, mul2(fy, fy)), a0, a1);
            if (fminf(a0, a1) <= thr32) {
                if (a0 <= thr32) exact(t);
                if (a1 <= thr32 && t + 1 < lim) exact(t + 1);
            }
        }
    }
    if (i >= n) return;
    const size_t o = (size_t)m[M_KPART_OFF] + ((size_t)slice * n + i) * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) { part_d2[o + k] = best[k]; part_idx[o + k] = bidx[k]; }
}

__global__ void __launch_bounds__(KNN_THREADS)
dmap_knn_merge_batch_kernel(const double* __restrict__ part_d2, const int32_t* __restrict__ part_idx,
                            const int64_t* __restrict__ meta, int n_images, int total_heads, int max_slices,
                            int32_t* __restrict__ nn_idx, double* __restrict__ nn_dist, double* __restrict__ sigma) {
    const int g = blockIdx.x * KNN_THREADS + threadIdx.x;
    if (g >= total_heads) return;
    const int img = find_image(meta, n_images + 1, M_PT_OFF, g);
    const int64_t* m = meta + (size_t)img * META_COLS;
    const int n = (int)m[M_N], i = g - (int)m[M_PT_OFF];
    const int slices = knn_slicing(n, max_slices).slices();
    double best[4];
    int bidx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { best[k] = INFINITY; bidx[k] = n; }
    for (int s = 0; s < slices; ++s) {
        const size_t o = (size_t)m[M_KPART_OFF] + ((size_t)s * n + i) * 4;
        for (int k = 0; k < 4; ++k) {
            const double d2 = part_d2[o + k];
            const int j = part_idx[o + k];
            if (j < n && (d2 < best[3] || (d2 == best[3] && j < bidx[3]))) knn_insert(best, bidx, d2, j);
        }
    }
    double d[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        d[k] = __dsqrt_rn(best[k]);
        if (nn_idx) nn_idx[4 * (size_t)g + k] = bidx[k];
        if (nn_dist) nn_dist[4 * (size_t)g + k] = d[k];
    }
    sigma[g] = (n > 3) ? __dmul_rn(__dadd_rn(__dadd_rn(d[1], d[2]), d[3]), 0.1) : 15.0;
}

// ---------------------------------------------------------------------------------- prepare
constexpr int PREP_WARPS = 4;

// Shape of scipy's 1-D kernel for one sigma, evaluated by a whole warp (all lanes return the same values):
// radius int(truncate*sigma + 0.5), coef -0.5/sigma^2 and the normaliser in numpy's pairwise order.
__device__ void stamp_shape(double sd, double truncate, LeafList& ll, int lane, int& radius, double& coef, double& norm) {
    if (!(sd > 1e-15)) {  // scipy: sigma <= 1e-15 copies the input (identity filter)
        radius = 0; coef = 0.0; norm = 1.0;
        return;
    }
    // scipy: int(truncate * float(sigma) + 0.5); clamped far beyond any image so that box arithmetic cannot
    // overflow (a radius that large covers every pixel anyway, the weights use coef / norm)
    const double rd = __dadd_rn(__dmul_rn(truncate, sd), 0.5);
    radius = rd < 1.0e9 ? (int)rd : 1000000000;
    coef = -0.5 / __dmul_rn(sd, sd);
    const int n_el = 2 * radius + 1;
    const int n_leaves = enumerate_leaves(-radius, n_el, ll, lane == 0);
    double v;
    if (n_leaves < 0) {
        v = (lane == 0) ? pairwise_phi_sum(coef, -radius, n_el) : 0.0;  // absurdly wide kernel
    } else {
        __syncwarp();
        const int group = lane >> 3, sub = lane & 7;
        const unsigned group_mask = 0xffu << (8 * group);
        for (int l0 = 0; l0 < n_leaves; l0 += 4) {
            const int l = l0 + group;
            if (l < n_leaves) {  // uniform inside a group of 8 lanes
                const double lv = leaf_by_group(coef, ll.first[l], ll.len[l], sub, group_mask);
                if (sub == 0) ll.sum[l] = lv;
            }
        }
        __syncwarp();
        v = (lane == 0) ? combine_leaves(-radius, n_el, ll) : 0.0;
    }
    norm = __shfl_sync(FULL_MASK, v, 0);
}

// Pixel of the one-hot write and the skip test of dmap_gen.py:41-44; false = the head is skipped.
__device__ __forceinline__ bool stamp_pixel(double2 p, int height, int width, int& ix, int& iy) {
    ix = (int)p.x;  // Python int(): truncation toward zero
    iy = (int)p.y;
    const bool keep = iy < height && ix < width;
    if (iy < 0) iy += height;  // numpy wraps negative indices; the host wrapper rejects < -size like numpy
    if (ix < 0) ix += width;
    return keep && iy >= 0 && ix >= 0;
}

__device__ __forceinline__ int4 stamp_box(int ix, int iy, int radius) {
    return radius < 0 ? make_int4(1, 0, 1, 0)
                      : make_int4(max(ix - radius, -(1 << 30)), min(ix + radius, 1 << 30),
                                  max(iy - radius, -(1 << 30)), min(iy + radius, 1 << 30));
}

// Occupancy bitmap, one bit per fine tile of the batch: set for every tile the stamp's box touches.  Tiles whose
// bit stays clear are written as zeros by the splat kernel without looking at any list.  `step` lanes share the loop.
__device__ __forceinline__ void mark_tiles(const int4 b, int height, int width, int64_t ftile_off,
                                           unsigned* __restrict__ fmask, int first, int step) {
    if (b.x > b.y) return;
    const int tx0 = max(b.x, 0) / FINE_W, tx1 = min(b.y, width - 1) / FINE_W;
    const int ty0 = max(b.z, 0) / FINE_H, ty1 = min(b.w, height - 1) / FINE_H;
    if (tx1 < tx0 || ty1 < ty0) return;
    const int nx = tx1 - tx0 + 1, total = nx * (ty1 - ty0 + 1), ftx = ceil_div(width, FINE_W);
    for (int k = first; k < total; k += step) {
        const int64_t g = ftile_off + (int64_t)(ty0 + k / nx) * ftx + tx0 + k % nx;
        const unsigned bit = 1u << (g & 31);
        if (!(fmask[g >> 5] & bit)) atomicOr(fmask + (g >> 5), bit);  // mostly already set in a crowd
    }
}

// Adaptive sigma: one warp per head of the whole batch.  Writes the Stamp (weights), the Box (bounding box of
// the stamp, the only thing the culling passes read; an empty box marks a skipped head), the weight table of
// narrow stamps (radius < TAB, every head of a dense crowd: the normalised 1-D weights w[|d|] are tabulated
// once here instead of being re-evaluated -- fp64 exp + division -- by every tile the stamp touches) and the
// tile occupancy bits.
__global__ void __launch_bounds__(PREP_WARPS * 32)
dmap_prepare_kernel(const double2* __restrict__ pts, const double* __restrict__ sigma, double truncate,
                    const int64_t* __restrict__ meta, int n_images, int total_heads, Stamp* __restrict__ stamps,
                    int4* __restrict__ boxes, double* __restrict__ wtab, unsigned* __restrict__ fmask) {
    __shared__ LeafList leaves[PREP_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * PREP_WARPS + warp;
    if (i >= total_heads) return;
    const int img = find_image(meta, n_images + 1, M_PT_OFF, i);
    const int64_t* m = meta + (size_t)img * META_COLS;
    const int height = (int)__ldg(m + M_H), width = (int)__ldg(m + M_W);
    Stamp s;
    s.pad_ = 0;
    if (!stamp_pixel(pts[i], height, width, s.ix, s.iy)) {
        s.radius = -1; s.coef = 0.0; s.norm = 1.0;
    } else {
        stamp_shape(sigma[i], truncate, leaves[warp], lane, s.radius, s.coef, s.norm);
    }
    if (s.radius >= 0 && s.radius < TAB && lane <= s.radius)
        wtab[(size_t)i * TAB + lane] = __ddiv_rn(phi(s.coef, lane), s.norm);
    const int4 box = stamp_box(s.ix, s.iy, s.radius);
    if (lane == 0) {
        stamps[i] = s;
        boxes[i] = box;
    }
    mark_tiles(box, height, width, __ldg(m + M_FTILE_OFF), fmask, lane, 32);
}

// Fixed sigma: every stamp has the same shape, so one warp evaluates it once (template Stamp + weight table) ...
__global__ void __launch_bounds__(32)
dmap_fixed_template_kernel(double fixed_sigma, double truncate, Stamp* __restrict__ tmpl, double* __restrict__ tmpl_tab) {
    __shared__ LeafList ll;
    const int lane = threadIdx.x;
    Stamp s;
    s.ix = s.iy = 0; s.pad_ = 0;
    stamp_shape(fixed_sigma, truncate, ll, lane, s.radius, s.coef, s.norm);
    tmpl_tab[lane] = (lane <= s.radius && s.radius < TAB) ? __ddiv_rn(phi(s.coef, lane), s.norm) : 0.0;
    if (lane == 0) *tmpl = s;
}

// ... and one thread per head fills in the position.
__global__ void __launch_bounds__(256)
dmap_prepare_fixed_kernel(const double2* __restrict__ pts, const Stamp* __restrict__ tmpl,
                          const int64_t* __restrict__ meta, int n_images,
                          int total_heads, Stamp* __restrict__ stamps, int4* __restrict__ boxes,
                          unsigned* __restrict__ fmask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total_heads) return;
    const int img = find_image(meta, n_images + 1, M_PT_OFF, i);
    const int64_t* m = meta + (size_t)img * META_COLS;
    const int height = (int)__ldg(m + M_H), width = (int)__ldg(m + M_W);
    Stamp s = *tmpl;
    const int radius = s.radius;
    if (!stamp_pixel(pts[i], height, width, s.ix, s.iy)) {
        s.radius = -1; s.coef = 0.0; s.norm = 1.0;
    }  // no per-head weight table: the splat reads the template's (shared_tab)
    const int4 box = stamp_box(s.ix, s.iy, s.radius);
    stamps[i] = s;
    boxes[i] = box;
    mark_tiles(box, height, width, __ldg(m + M_FTILE_OFF), fmask, 0, 1);
}

// --------------------------------------------------------------------- two-level culling + splat
__device__ __forceinline__ bool box_hits(const int4 b, int x0, int y0, int w, int h) {
    return b.x <= b.y && b.y >= x0 && b.x < x0 + w && b.w >= y0 && b.z < y0 + h;
}

// Ordered compaction of one flag per thread across a CTA of THREADS; returns the slot of a set flag
// and the CTA total.  Two __syncthreads; warp_cnt is reused by the next call only after a later barrier.
template <int THREADS>
__device__ __forceinline__ int cta_compact(bool hit, int* warp_cnt, int& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned ballot = __ballot_sync(FULL_MASK, hit);
    __syncthreads();  // previous readers of warp_cnt are done
    if (lane == 0) warp_cnt[warp] = __popc(ballot);
    __syncthreads();
    int before = 0;
    total = 0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) {
        const int c = warp_cnt[w];
        if (w < warp) before += c;
        total += c;
    }
    return before + __popc(ballot & ((1u << lane) - 1u));
}

// Coarse pass.  Task = (image, coarse tile, chunk of CHUNK heads).  WRITE = false counts the chunk's heads
// whose box touches the coarse tile; WRITE = true repeats the scan and writes their indices, in index order,
// behind the heads of the lower chunks (counts summed on the fly), so that every coarse tile ends up with one
// contiguous ordered list; the last chunk also stores the list's length.
template <bool WRITE, bool PACKED = false>
__global__ void __launch_bounds__(COARSE_THREADS)
dmap_coarse_kernel(const int4* __restrict__ boxes, const int64_t* __restrict__ meta, int n_images,
                   int32_t* __restrict__ ccount, int32_t* __restrict__ ctotal, int32_t* __restrict__ clist) {
    __shared__ int warp_cnt[COARSE_THREADS / 32];
    const int img = find_image(meta, n_images + 1, M_CTASK_OFF, blockIdx.x);
    const int64_t* m = meta + (size_t)img * META_COLS;
    const int n = (int)m[M_N], width = (int)m[M_W];
    const int nchunks = ceil_div(n, CHUNK), ctx = ceil_div(width, COARSE);
    const int local = blockIdx.x - (int)m[M_CTASK_OFF];
    const int chunk = local % nchunks, ct = local / nchunks;
    DGVCC_DEV_CHECK(img >= 0 && img < n_images && n > 0 && local >= 0 && ct < ctx * ceil_div((int)m[M_H], COARSE));
    const int x0 = (ct % ctx) * COARSE, y0 = (ct / ctx) * COARSE;
    const int4* b = boxes + m[M_PT_OFF];
    int32_t* cnt_row = ccount + m[M_CTASK_OFF] + (size_t)ct * nchunks;
    int pos = 0;
    int32_t* out = nullptr;
    if (WRITE) {
        for (int c = 0; c < chunk; ++c) pos += cnt_row[c];
        out = clist + m[M_CLIST_OFF] + (size_t)ct * n;
    }
    const int i_end = min(n, (chunk + 1) * CHUNK);
    int count = 0;
    for (int base = chunk * CHUNK; base < i_end; base += COARSE_THREADS) {
        const int i = base + threadIdx.x;
        const int4 bi = i < i_end ? __ldg(b + i) : make_int4(1, 0, 1, 0);
        const bool hit = i < i_end && box_hits(bi, x0, y0, COARSE, COARSE);
        int total;
        const int slot = cta_compact<COARSE_THREADS>(hit, warp_cnt, total);
        // PACKED (fixed sigma, identical stamps): the list carries the stamp's centre pixel (row << 16 | column) instead
        // of the head index -- the fine pass needs nothing else and saves the dependent loads through the index
        DGVCC_DEV_CHECK(!(WRITE && hit) || (pos + count + slot >= 0 && pos + count + slot < n));
        if (WRITE && hit) out[pos + count + slot] = PACKED ? (int)(((unsigned)((bi.z + bi.w) >> 1) << 16) | (unsigned)((bi.x + bi.y) >> 1)) : i;
        count += total;
    }
    if (threadIdx.x == 0) {
        if (!WRITE) cnt_row[chunk] = count;
        else if (chunk == nchunks - 1) ctotal[m[M_CTILE_OFF] + ct] = pos + count;
    }
}

// Fine pass: one CTA (4 warps) per 32 x 32 output tile; warp w owns the band of rows [8w, 8w + 8), lane = column.
// Warp 0 decodes the tile (image, position, length of the coarse list) once for the CTA.  A tile whose
// occupancy bit is clear stores zeros at once.  Otherwise the CTA walks the ordered list of its coarse tile and
// keeps the heads whose stamp touches the fine tile (ordered compaction again).  Heads are staged GROUP at a
// time: narrow stamps copy their weight table w[|d|] (and its fl32-rounded twin), wide ones (at most GEN_MAX
// per group) get their 32 row and 32 column weights evaluated for this tile.  Each warp then picks, by ballot,
// the staged heads that reach its band and accumulates fl32(f64(fl32(wy)) * wx) per pixel in fp32, in head
// order.  Rows and columns a stamp does not reach add (float)(0 * w) = +0, which changes nothing (the sums are
// never -0), so they are skipped.  Every pixel of the packed output is written exactly once, coalesced; zero
// fill fused.
struct __align__(16) TileDesc {  // 64 bytes, written by dmap_tile_setup_kernel, read whole by every thread of the tile's CTA
    int x0, y0, width, height;
    int cnt, n, pad0_, pad1_;      // cnt: length of the coarse tile's list, 0 when no stamp touches the fine tile
    long long out_off, clist_off;
    long long pt_off, pad2_;
};
static_assert(sizeof(TileDesc) == 64, "TileDesc is read as four 16-byte words");

// One thread per fine tile of the batch: image lookup, tile position, occupancy bit, coarse-list length.
__global__ void __launch_bounds__(256)
dmap_tile_setup_kernel(const int64_t* __restrict__ meta, int n_images, int fine_tiles, const unsigned* __restrict__ fmask,
                       const int32_t* __restrict__ ctotal, int have_heads, TileDesc* __restrict__ desc) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= fine_tiles) return;
    const int img = find_image(meta, n_images + 1, M_FTILE_OFF, t);
    const int64_t* m = meta + (size_t)img * META_COLS;
    TileDesc d;
    d.n = (int)m[M_N]; d.height = (int)m[M_H]; d.width = (int)m[M_W];
    const int ftx = ceil_div(d.width, FINE_W);
    const int local = t - (int)m[M_FTILE_OFF];
    DGVCC_DEV_CHECK(img >= 0 && img < n_images && local >= 0 && local < ftx * ceil_div(d.height, FINE_H));
    d.x0 = (local % ftx) * FINE_W; d.y0 = (local / ftx) * FINE_H;
    d.pt_off = m[M_PT_OFF]; d.out_off = m[M_OUT_OFF];
    d.cnt = 0; d.clist_off = 0; d.pad0_ = d.pad1_ = 0; d.pad2_ = 0;
    if (have_heads && d.n > 0 && ((fmask[t >> 5] >> (t & 31)) & 1u)) {
        const int ct = (d.y0 / COARSE) * ceil_div(d.width, COARSE) + d.x0 / COARSE;
        d.cnt = ctotal[m[M_CTILE_OFF] + ct];
        d.clist_off = m[M_CLIST_OFF] + (long long)ct * d.n;
    }
    desc[t] = d;
}

__global__ void __launch_bounds__(SPLAT_THREADS, 9)
dmap_splat_kernel(const Stamp* __restrict__ stamps, const double* __restrict__ wtab, const int4* __restrict__ boxes,
                  const TileDesc* __restrict__ desc, const int32_t* __restrict__ clist,
                  const double* __restrict__ shared_tab, float* __restrict__ density) {
    __shared__ int list[SPLAT_THREADS];
    __shared__ int4 lbox[SPLAT_THREADS];     // boxes of the listed heads
    __shared__ int warp_cnt[SPLAT_THREADS / 32];
    __shared__ double tab[GROUP][TAB];       // w[|d|]
    __shared__ double tabf[GROUP][TAB];      // (double)(float)w[|d|]: the first filter pass stores float32
    __shared__ double gwy[GEN_MAX][FINE_H];  // wide stamps: fl32-rounded row weights, widened again (exact)
    __shared__ double gwx[GEN_MAX][FINE_W];
    __shared__ int gen_head[GEN_MAX];
    __shared__ double stab[2][TAB];          // fixed sigma: the one table every narrow stamp shares, and its fl32 twin

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (shared_tab && tid < TAB) {
        const double w = __ldg(shared_tab + tid);
        stab[0][tid] = w;
        stab[1][tid] = (double)(float)w;
    }  // ordered before its first use by the barriers of the list scan
    const int4* dp = reinterpret_cast<const int4*>(desc + blockIdx.x);
    const int4 d0 = __ldg(dp), d1 = __ldg(dp + 1);
    const longlong2 d2 = __ldg(reinterpret_cast<const longlong2*>(dp + 2));
    const int x0 = d0.x, y0 = d0.y, width = d0.z, height = d0.w, cnt = d1.x;
    const int yb = y0 + SPLAT_RPT * warp;  // first row of this warp's band
    const int x = x0 + lane;
    DGVCC_DEV_CHECK(x0 >= 0 && y0 >= 0 && x0 < width && y0 < height && cnt >= 0 && d2.x >= 0 && d2.y >= 0);
    float acc[SPLAT_RPT];  // pixels (yb + k, x)
#pragma unroll
    for (int k = 0; k < SPLAT_RPT; ++k) acc[k] = 0.f;

    if (cnt > 0) {
        const long long pt_off = __ldg(reinterpret_cast<const long long*>(dp + 3));
        const int32_t* cl = clist + d2.y;
        const int4* bx = boxes + pt_off;
        const Stamp* st = stamps + pt_off;
        const double* wt = wtab + (size_t)pt_off * TAB;
        for (int base = 0; base < cnt; base += SPLAT_THREADS) {
            int i = -1;
            int4 b = make_int4(1, 0, 1, 0);
            bool hit = false;
            if (base + tid < cnt) {
                i = __ldg(cl + base + tid);
                DGVCC_DEV_CHECK(i >= 0);
                b = __ldg(bx + i);
                hit = box_hits(b, x0, y0, FINE_W, FINE_H);
            }
            int total;
            const int slot = cta_compact<SPLAT_THREADS>(hit, warp_cnt, total);
            if (hit) { list[slot] = i; lbox[slot] = b; }
            __syncthreads();
            for (int c0 = 0; c0 < total; c0 += GROUP) {
                const int ccnt = min(GROUP, total - c0);
                // which heads of the chunk are wide (a box narrower than 2*TAB cannot be a clamped one, so centre
                // and radius of narrow stamps follow from the box)
                unsigned long long wide_mask = 0;
#pragma unroll
                for (int w = 0; w < GROUP / 32; ++w) {
                    const int t = 32 * w + lane;
                    const bool wide = t < ccnt && (lbox[c0 + t].y - lbox[c0 + t].x) >= 2 * TAB;
                    wide_mask |= (unsigned long long)__ballot_sync(FULL_MASK, wide) << (32 * w);
                }
                // a chunk with few wide heads is one group; otherwise groups of GEN_MAX heads
                const int gs = __popcll(wide_mask) <= GEN_MAX ? GROUP : GEN_MAX;
                for (int g0 = 0; g0 < ccnt; g0 += gs) {
                    const int g1 = min(ccnt, g0 + gs);
                    const unsigned long long range = (g1 - g0 == 64) ? ~0ull : (((1ull << (g1 - g0)) - 1ull) << g0);
                    const unsigned long long wide_here = wide_mask & range;
                    const int n_wide = __popcll(wide_here);
                    // narrow heads: copy the weight tables (a warp reads one head's table per step, all of its
                    // steps in flight together); with a shared table (fixed sigma) there is nothing to copy
                    if (!shared_tab) {
                        double wv[GROUP / SPLAT_WARPS];
#pragma unroll
                        for (int u = 0; u < GROUP / SPLAT_WARPS; ++u) {
                            const int t = g0 + warp + u * SPLAT_WARPS;
                            wv[u] = 0.0;
                            if (t < g1) {
                                const int r = (lbox[c0 + t].y - lbox[c0 + t].x) >> 1;
                                if (lane <= r && r < TAB) wv[u] = __ldg(wt + (size_t)list[c0 + t] * TAB + lane);
                            }
                        }
#pragma unroll
                        for (int u = 0; u < GROUP / SPLAT_WARPS; ++u) {
                            const int t = g0 + warp + u * SPLAT_WARPS;
                            if (t < g1) {  // entries past the radius are never read
                                tab[t][lane] = wv[u];
                                tabf[t][lane] = (double)(float)wv[u];
                            }
                        }
                    }
                    if (tid >= g0 && tid < g1 && ((wide_mask >> tid) & 1ull))
                        gen_head[__popcll(wide_here & ((1ull << tid) - 1ull))] = tid;
                    if (n_wide) {
                        __syncthreads();
                        for (int k = tid; k < n_wide * (FINE_H + FINE_W); k += SPLAT_THREADS) {
                            const int gsl = k / (FINE_H + FINE_W), off = k % (FINE_H + FINE_W);
                            const Stamp s = st[list[c0 + gen_head[gsl]]];
                            const bool is_x = off >= FINE_H;
                            const int d = is_x ? (x0 + off - FINE_H - s.ix) : (y0 + off - s.iy);
                            double w = 0.0;
                            if (d >= -s.radius && d <= s.radius) w = __ddiv_rn(phi(s.coef, d), s.norm);
                            if (is_x) gwx[gsl][off - FINE_H] = w;
                            else gwy[gsl][off] = (double)(float)w;
                        }
                    }
                    __syncthreads();
                    // accumulate, in head order, the staged heads that reach this warp's band
                    for (int j0 = g0; j0 < g1; j0 += 32) {
                        const int t = j0 + lane;
                        bool reach = false;
                        if (t < g1) {
                            const int4 b = lbox[c0 + t];
                            reach = b.w >= yb && b.z < yb + SPLAT_RPT;
                        }
                        unsigned todo = __ballot_sync(FULL_MASK, reach);
                        while (todo) {
                            const int hd = j0 + __ffs(todo) - 1;
                            todo &= todo - 1;
                            const int4 b = lbox[c0 + hd];
                            const int r = (b.y - b.x) >> 1;
                            if (r < TAB) {
                                const int dx = abs(x - ((b.x + b.y) >> 1));
                                if (__any_sync(FULL_MASK, dx <= r)) {
                                    const double* tb = shared_tab ? stab[0] : tab[hd];
                                    const double* tbf = shared_tab ? stab[1] : tabf[hd];
                                    const double cx = dx <= r ? tb[dx] : 0.0;
                                    const int dy0 = yb - ((b.z + b.w) >> 1);
#pragma unroll
                                    for (int k = 0; k < SPLAT_RPT; ++k) {
                                        const int dy = abs(dy0 + k);
                                        if (dy <= r)  // warp-uniform
                                            acc[k] = __fadd_rn(acc[k], (float)__dmul_rn(tbf[dy], cx));
                                    }
                                }
                            } else {
                                const int gsl = __popcll(wide_here & ((1ull << hd) - 1ull));
                                const double cx = gwx[gsl][lane];
#pragma unroll
                                for (int k = 0; k < SPLAT_RPT; ++k) {
                                    const double ry = gwy[gsl][SPLAT_RPT * warp + k];
                                    if (ry != 0.0) acc[k] = __fadd_rn(acc[k], (float)__dmul_rn(ry, cx));  // warp-uniform
                                }
                            }
                        }
                    }
                    __syncthreads();
                }
            }
        }
    }
    if (x < width && yb < height) {
        float* out = density + d2.x + (size_t)yb * width + x;
        if (yb + SPLAT_RPT <= height) {
#pragma unroll
            for (int k = 0; k < SPLAT_RPT; ++k) out[(size_t)k * width] = acc[k];
        } else {
#pragma unroll
            for (int k = 0; k < SPLAT_RPT; ++k)
                if (yb + k < height) out[(size_t)k * width] = acc[k];
        }
    }
}

// ------------------------------------------------------------------------------- fixed sigma, 15 x 15 stamps
// gaussian_filter_density_fixed (dmap_gen.py:53-81; what run() calls): sigma 4, truncate 7/4 -> radius 7, every head
// adds the SAME 15 x 15 table fl32(f64(fl32(w[|dy|])) * w[|dx|]), only shifted.  One WARP owns one 32 x 32 output tile:
//   * accumulators in shared memory with an apron of R pixels on every side (46 x 46; 8.7 KB per warp, so that 24
//     warps fit an SM -- a 2R apron needs no clipping tests at all but allows only 12, and the kernel is bound by
//     memory latency, not by instruction issue); stamp pixels beyond the apron are predicated off; only the inner
//     32 x 32 is stored;
//   * the 225 stamp pixels are spread over the lanes (7 full steps + one pixel): lane l step k handles stamp pixel
//     p = 32 k + l, whose table value and offset inside the apron tile sit in registers for the life of the warp --
//     per stamp and step: the apron test, LDS, FADD, STS (the row pitch 47 = 15 mod 32 makes the 32 lanes
//     of a step hit 32 different banks);
//   * stamps are applied in list order, one after the other, by the same warp: every pixel sees its heads in index
//     order, which is what makes the fp32 sums bit-identical to the reference's sequential accumulation;
//   * the list of the coarse tile carries packed centre pixels (dmap_coarse_kernel<true, true>): one coalesced load
//     per 32 entries, the next one already in flight.
// Against dmap_splat_kernel (lane = tile column, 8 rows per thread, 105 instructions per 8-row band and stamp with
// half the lanes idle on a 15-wide stamp) this is ~45 instructions per (tile, stamp) with every lane busy.
constexpr int FAST_R = 7;
constexpr int FAST_S = 2 * FAST_R + 1;             // 15
constexpr int FAST_APRON = 32 + 2 * FAST_R;        // 46: apron of R pixels; stamp pixels beyond it are predicated off
constexpr int FAST_PITCH = 47;                     // >= FAST_APRON, = FAST_S (mod 32)
constexpr int FAST_TILE_FLOATS = (FAST_APRON * FAST_PITCH + 3) / 4 * 4;   // 2164 floats = 8656 bytes per warp
constexpr int FAST_STEPS = (FAST_S * FAST_S + 31) / 32;     // 8; the last one holds a single pixel
constexpr int FAST_SMEM = SPLAT_WARPS * FAST_TILE_FLOATS * 4;
static_assert(FAST_S * FAST_S == 32 * (FAST_STEPS - 1) + 1, "layout of the 15 x 15 stamp over the lanes");

__global__ void __launch_bounds__(256)
dmap_fixed_table_kernel(const double* __restrict__ tmpl_tab, float* __restrict__ tab2d) {
    const int p = threadIdx.x;
    if (p >= FAST_S * FAST_S) return;
    const int dy = abs(p / FAST_S - FAST_R), dx = abs(p % FAST_S - FAST_R);
    // the first pass of the separable filter stores float32, the second multiplies in double and stores float32
    tab2d[p] = (float)__dmul_rn((double)(float)tmpl_tab[dy], tmpl_tab[dx]);
}

// Fast-path prepare: the box of every head (the only thing the culling passes read) and the tile occupancy bits.
__global__ void __launch_bounds__(256)
dmap_prepare_fast_kernel(const double2* __restrict__ pts, const int64_t* __restrict__ meta, int n_images, int total_heads,
                         int4* __restrict__ boxes, unsigned* __restrict__ fmask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total_heads) return;
    const int img = find_image(meta, n_images + 1, M_PT_OFF, i);
    const int64_t* m = meta + (size_t)img * META_COLS;
    const int height = (int)__ldg(m + M_H), width = (int)__ldg(m + M_W);
    int ix, iy;
    const bool keep = stamp_pixel(pts[i], height, width, ix, iy);
    const int4 box = stamp_box(ix, iy, keep ? FAST_R : -1);
    boxes[i] = box;
    mark_tiles(box, height, width, __ldg(m + M_FTILE_OFF), fmask, 0, 1);
}

__global__ void __launch_bounds__(SPLAT_THREADS)
dmap_splat_fixed_kernel(const TileDesc* __restrict__ desc, int fine_tiles, const unsigned* __restrict__ clist,
                        const float* __restrict__ tab2d, float* __restrict__ density) {
    extern __shared__ float4 fast_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = blockIdx.x * SPLAT_WARPS + warp;
    if (t >= fine_tiles) return;  // warps never synchronise with each other
    float* tile = reinterpret_cast<float*>(fast_smem) + warp * FAST_TILE_FLOATS;
    const int4* dp = reinterpret_cast<const int4*>(desc + t);
    const int4 d0 = __ldg(dp), d1 = __ldg(dp + 1);
    const longlong2 d2 = __ldg(reinterpret_cast<const longlong2*>(dp + 2));
    const int x0 = d0.x, y0 = d0.y, width = d0.z, height = d0.w, cnt = d1.x;
    const int x = x0 + lane;
    DGVCC_DEV_CHECK(x0 >= 0 && y0 >= 0 && x0 < width && y0 < height && cnt >= 0 && d2.x >= 0 && d2.y >= 0);
    float* out = density + d2.x + (size_t)y0 * width + x;
    const int rows = min(FINE_H, height - y0);
    if (cnt == 0) {  // no stamp touches the tile
        if (x < width)
            for (int r = 0; r < rows; ++r) out[(size_t)r * width] = 0.f;
        return;
    }
    float tv[FAST_STEPS];
    int off[FAST_STEPS], dxy[FAST_STEPS];   // dxy: (row << 8 | column) of the stamp pixel inside the stamp
#pragma unroll
    for (int k = 0; k < FAST_STEPS; ++k) {
        const int p = min(32 * k + lane, FAST_S * FAST_S - 1);
        tv[k] = __ldg(tab2d + p);
        off[k] = (p / FAST_S) * FAST_PITCH + p % FAST_S;
        dxy[k] = ((p / FAST_S) << 8) | (p % FAST_S);
    }
    float4* tile4 = reinterpret_cast<float4*>(tile);
    for (int i = lane; i < FAST_TILE_FLOATS / 4; i += 32) tile4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncwarp();
    const unsigned* cl = clist + d2.y;
    // the scan of the coarse tile's list is a chain of L2 round trips: four batches of 32 entries are in flight at a time
    constexpr int AHEAD = 4;
    unsigned nxt[AHEAD];
#pragma unroll
    for (int q = 0; q < AHEAD; ++q) nxt[q] = 32 * q + lane < cnt ? __ldg(cl + 32 * q + lane) : 0xffffffffu;
    for (int base0 = 0; base0 < cnt; base0 += 32 * AHEAD) {
        unsigned cur[AHEAD];
#pragma unroll
        for (int q = 0; q < AHEAD; ++q) {
            cur[q] = nxt[q];
            const int j = base0 + 32 * (AHEAD + q) + lane;
            nxt[q] = j < cnt ? __ldg(cl + j) : 0xffffffffu;
        }
#pragma unroll
        for (int q = 0; q < AHEAD; ++q) {
        const int base = base0 + 32 * q;
        const unsigned e = cur[q];
        const int ix = (int)(e & 0xffffu), iy = (int)(e >> 16);
        const bool hit = base + lane < cnt && ix + FAST_R >= x0 && ix - FAST_R < x0 + FINE_W && iy + FAST_R >= y0 &&
                         iy - FAST_R < y0 + FINE_H;
        unsigned todo = __ballot_sync(FULL_MASK, hit);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const unsigned s = __shfl_sync(FULL_MASK, e, src);
            // top-left pixel of the stamp relative to the apron tile (whose origin is the tile's minus R): -R .. 31 + R
            const int ay = (int)(s >> 16) - y0, ax = (int)(s & 0xffffu) - x0;
            float* a = tile + ay * FAST_PITCH + ax;
            float v[FAST_STEPS];
            bool in[FAST_STEPS];
#pragma unroll
            for (int k = 0; k < FAST_STEPS; ++k) {   // 32 different pixels per step; those beyond the apron are nobody's
                in[k] = (unsigned)(ay + (dxy[k] >> 8)) < (unsigned)FAST_APRON && (unsigned)(ax + (dxy[k] & 255)) < (unsigned)FAST_APRON &&
                        (k < FAST_STEPS - 1 || lane == 0);   // the last step holds pixel 224 only
                DGVCC_DEV_CHECK(!in[k] || (a + off[k] >= tile && a + off[k] < tile + FAST_TILE_FLOATS));
                v[k] = in[k] ? a[off[k]] : 0.f;
            }
#pragma unroll
            for (int k = 0; k < FAST_STEPS; ++k)
                if (in[k]) a[off[k]] = __fadd_rn(v[k], tv[k]);
            __syncwarp();  // the next stamp may touch the same pixels from other lanes
        }
        }
    }
    if (x < width) {
        const float* src = tile + FAST_R * FAST_PITCH + FAST_R + lane;
        for (int r = 0; r < rows; ++r) out[(size_t)r * width] = src[r * FAST_PITCH];
    }
}

}  // namespace dmap
}  // namespace dgvcc

using namespace dgvcc;
using namespace dgvcc::dmap;

static int knn_slices(int n) {
    const int query_ctas = ceil_div(n, KNN_THREADS);
    int s = ceil_div(4 * 148, query_ctas);       // ~4 CTAs per SM in flight
    const int max_s = ceil_div(n, KNN_THREADS);  // a slice is at least one candidate tile
    if (s > max_s) s = max_s;
    return s < 1 ? 1 : s;
}

extern "C" size_t dgvcc_dmap_knn_workspace_bytes(int n) {
    if (n <= 0) return 16;
    return (size_t)knn_slices(n) * n * 4 * (sizeof(double) + sizeof(int32_t));
}

extern "C" int dgvcc_dmap_knn_sigma(const double* pts_xy, int n, int32_t* nn_idx, double* nn_dist, double* sigma,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (n < 0) return DGVCC_ERR_ARG;
    if (n == 0) return DGVCC_OK;
    if (!pts_xy || !nn_idx || !nn_dist || !sigma || !workspace) return DGVCC_ERR_ARG;
    if (workspace_bytes < dgvcc_dmap_knn_workspace_bytes(n)) return DGVCC_ERR_WORKSPACE;
    const int slices = knn_slices(n);
    const int slice_len = ceil_div(ceil_div(n, slices), KNN_THREADS) * KNN_THREADS;
    const int used = ceil_div(n, slice_len);
    double* part_d2 = (double*)workspace;
    int32_t* part_idx = (int32_t*)(part_d2 + (size_t)slices * n * 4);
    cudaStream_t st = (cudaStream_t)stream;
    dmap_knn_kernel<<<dim3(ceil_div(n, KNN_THREADS), used), KNN_THREADS, 0, st>>>((const double2*)pts_xy, n, slice_len,
                                                                                 part_d2, part_idx);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    dmap_knn_merge_kernel<<<ceil_div(n, KNN_THREADS), KNN_THREADS, 0, st>>>(part_d2, part_idx, n, used, nn_idx, nn_dist, sigma);
    return (int)cudaGetLastError();
}

// ---- batch plan (host only) ---------------------------------------------------------------------
extern "C" int dgvcc_dmap_batch_plan(int n_images, const int32_t* heights, const int32_t* widths, const int32_t* counts,
                                     int64_t* meta, dgvcc_dmap_plan* plan) {
    int64_t max_side = 0;
    if (n_images <= 0 || !heights || !widths || !counts || !meta || !plan) return DGVCC_ERR_ARG;
    int64_t acc[META_COLS] = {0};
    // kNN: as many candidate slices per image as it takes to fill the chip with tasks, no more
    int64_t query_blocks = 0;
    for (int i = 0; i < n_images; ++i) query_blocks += counts[i] > 0 ? ceil_div(counts[i], KNN_THREADS) : 0;
    int max_slices = query_blocks > 0 ? (int)((148 * 8 + query_blocks - 1) / query_blocks) : 1;
    if (max_slices > 64) max_slices = 64;
    plan->knn_max_slices = max_slices;
    for (int i = 0; i <= n_images; ++i) {
        int64_t* m = meta + (size_t)i * META_COLS;
        m[M_PT_OFF] = acc[M_PT_OFF]; m[M_OUT_OFF] = acc[M_OUT_OFF]; m[M_FTILE_OFF] = acc[M_FTILE_OFF];
        m[M_CTASK_OFF] = acc[M_CTASK_OFF]; m[M_CLIST_OFF] = acc[M_CLIST_OFF]; m[M_CTILE_OFF] = acc[M_CTILE_OFF];
        m[M_KTASK_OFF] = acc[M_KTASK_OFF]; m[M_KPART_OFF] = acc[M_KPART_OFF]; m[M_KQB_OFF] = acc[M_KQB_OFF];
        if (i == n_images) { m[M_N] = m[M_H] = m[M_W] = 0; break; }
        const int64_t n = counts[i], h = heights[i], w = widths[i];
        if (n < 0 || h <= 0 || w <= 0) return DGVCC_ERR_ARG;
        m[M_N] = n; m[M_H] = h; m[M_W] = w;
        max_side = h > max_side ? h : max_side;
        max_side = w > max_side ? w : max_side;
        const int64_t ctiles = (int64_t)ceil_div((int)w, COARSE) * ceil_div((int)h, COARSE);
        const int64_t nchunks = ceil_div((int)n, CHUNK), slices = n > 0 ? knn_slicing((int)n, max_slices).slices() : 0;
        acc[M_PT_OFF] += n;
        acc[M_OUT_OFF] += h * w;
        acc[M_FTILE_OFF] += (int64_t)ceil_div((int)w, FINE_W) * ceil_div((int)h, FINE_H);
        acc[M_CTASK_OFF] += ctiles * nchunks;
        acc[M_CLIST_OFF] += ctiles * n;
        acc[M_CTILE_OFF] += ctiles;
        acc[M_KTASK_OFF] += (int64_t)ceil_div((int)n, KNN_THREADS) * slices;
        acc[M_KQB_OFF] += ceil_div((int)n, KNN_THREADS);
        acc[M_KPART_OFF] += slices * n * 4;
    }
    if (acc[M_FTILE_OFF] > 0x7fffffffLL || acc[M_CTASK_OFF] > 0x7fffffffLL || acc[M_KTASK_OFF] > 0x7fffffffLL ||
        acc[M_PT_OFF] > 0x7fffffffLL)
        return DGVCC_ERR_UNSUPPORTED;
    plan->max_side = max_side;
    plan->total_heads = acc[M_PT_OFF];
    plan->total_pixels = acc[M_OUT_OFF];
    plan->fine_tiles = acc[M_FTILE_OFF];
    plan->coarse_tasks = acc[M_CTASK_OFF];
    plan->knn_tasks = acc[M_KTASK_OFF];
    plan->knn_query_blocks = acc[M_KQB_OFF];
    size_t off = 0;
    const int64_t heads = acc[M_PT_OFF] > 0 ? acc[M_PT_OFF] : 1;
    plan->off_stamps = (int64_t)off; off = align_up(off + (size_t)heads * sizeof(Stamp), 256);
    plan->off_boxes = (int64_t)off;  off = align_up(off + (size_t)heads * sizeof(int4), 256);
    plan->off_wtab = (int64_t)off;   off = align_up(off + (size_t)heads * TAB * sizeof(double), 256);
    plan->off_fmask = (int64_t)off;  off = align_up(off + (size_t)(acc[M_FTILE_OFF] / 32 + 1) * 4, 256);
    plan->off_tmpl = (int64_t)off;   off = align_up(off + sizeof(Stamp) + TAB * sizeof(double) + 256 * sizeof(float), 256);
    plan->off_desc = (int64_t)off;   off = align_up(off + (size_t)acc[M_FTILE_OFF] * sizeof(TileDesc), 256);
    plan->off_ccount = (int64_t)off; off = align_up(off + (size_t)(acc[M_CTASK_OFF] + 1) * 4, 256);
    plan->off_ctotal = (int64_t)off; off = align_up(off + (size_t)(acc[M_CTILE_OFF] + 1) * 4, 256);
    plan->off_clist = (int64_t)off;  off = align_up(off + (size_t)(acc[M_CLIST_OFF] + 1) * 4, 256);
    plan->splat_workspace_bytes = (int64_t)off;
    off = 0;
    plan->off_knn_d2 = 0;            off = align_up((size_t)(acc[M_KPART_OFF] + 1) * 8, 256);
    plan->off_knn_idx = (int64_t)off; off = align_up(off + (size_t)(acc[M_KPART_OFF] + 1) * 4, 256);
    plan->off_knn_pts32 = (int64_t)off; off = align_up(off + (size_t)heads * sizeof(float2), 256);
    plan->off_knn_max = (int64_t)off; off = align_up(off + (size_t)n_images * sizeof(int), 256);
    plan->knn_workspace_bytes = (int64_t)off;
    return DGVCC_OK;
}

extern "C" int dgvcc_dmap_knn_sigma_batch(const double* pts_xy, int n_images, const int64_t* meta,
                                          const dgvcc_dmap_plan* plan, int32_t* nn_idx, double* nn_dist, double* sigma,
                                          void* workspace, size_t workspace_bytes, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (n_images <= 0 || !meta || !plan) return DGVCC_ERR_ARG;
    if (plan->total_heads == 0) return DGVCC_OK;
    if (!pts_xy || !sigma || !workspace) return DGVCC_ERR_ARG;
    if (workspace_bytes < (size_t)plan->knn_workspace_bytes) return DGVCC_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    double* part_d2 = (double*)((char*)workspace + plan->off_knn_d2);
    int32_t* part_idx = (int32_t*)((char*)workspace + plan->off_knn_idx);
    float2* pts32 = (float2*)((char*)workspace + plan->off_knn_pts32);
    int* img_max = (int*)((char*)workspace + plan->off_knn_max);
    const int heads = (int)plan->total_heads;
    DGVCC_RETURN_IF_CUDA(cudaMemsetAsync(img_max, 0, (size_t)n_images * sizeof(int), st));
    dmap_knn_prep_kernel<<<ceil_div(heads, 256), 256, 0, st>>>((const double2*)pts_xy, meta, n_images, heads, pts32, img_max);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    dmap_knn_batch_kernel<<<(unsigned)plan->knn_query_blocks, KNN_THREADS, 0, st>>>((const double2*)pts_xy, pts32, img_max, meta,
                                                                                    n_images, (int)plan->knn_max_slices, 0, part_d2,
                                                                                    part_idx);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    if (plan->knn_tasks > plan->knn_query_blocks) {
        dmap_knn_batch_kernel<<<(unsigned)(plan->knn_tasks - plan->knn_query_blocks), KNN_THREADS, 0, st>>>(
            (const double2*)pts_xy, pts32, img_max, meta, n_images, (int)plan->knn_max_slices, 1, part_d2, part_idx);
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    }
    dmap_knn_merge_batch_kernel<<<ceil_div((int)plan->total_heads, KNN_THREADS), KNN_THREADS, 0, st>>>(
        part_d2, part_idx, meta, n_images, (int)plan->total_heads, (int)plan->knn_max_slices, nn_idx, nn_dist, sigma);
    return (int)cudaGetLastError();
}

extern "C" int dgvcc_dmap_splat_batch(const double* pts_xy, const double* sigma, double fixed_sigma, double truncate,
                                      int n_images, const int64_t* meta, const dgvcc_dmap_plan* plan, void* workspace,
                                      size_t workspace_bytes, float* density, void* stream) {
    DGVCC_DEVICE_GUARD(stream);
    if (n_images <= 0 || !meta || !plan || !density || !workspace) return DGVCC_ERR_ARG;
    if (plan->total_heads > 0 && !pts_xy) return DGVCC_ERR_ARG;
    if (workspace_bytes < (size_t)plan->splat_workspace_bytes) return DGVCC_ERR_WORKSPACE;
    if (!sigma && !(fixed_sigma >= 0.0)) return DGVCC_ERR_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    Stamp* stamps = (Stamp*)(ws + plan->off_stamps);
    int4* boxes = (int4*)(ws + plan->off_boxes);
    double* wtab = (double*)(ws + plan->off_wtab);
    unsigned* fmask = (unsigned*)(ws + plan->off_fmask);
    Stamp* tmpl = (Stamp*)(ws + plan->off_tmpl);
    double* tmpl_tab = (double*)(ws + plan->off_tmpl + sizeof(Stamp));
    int32_t* ccount = (int32_t*)(ws + plan->off_ccount);
    int32_t* ctotal = (int32_t*)(ws + plan->off_ctotal);
    int32_t* clist = (int32_t*)(ws + plan->off_clist);
    const int heads = (int)plan->total_heads;
    // the reference's fixed generator (sigma 4, truncate 7/4: 15 x 15 stamps) takes the warp-per-tile kernel; its lists
    // pack the centre pixel into 16 + 16 bits
    const bool fast = !sigma && (int)(truncate * fixed_sigma + 0.5) == FAST_R && plan->max_side > 0 && plan->max_side < 65536;
    float* tab2d = (float*)(ws + plan->off_tmpl + sizeof(Stamp) + TAB * sizeof(double));
    if (heads > 0) {
        DGVCC_RETURN_IF_CUDA(cudaMemsetAsync(fmask, 0, (size_t)(plan->fine_tiles / 32 + 1) * 4, st));
        if (sigma) {
            dmap_prepare_kernel<<<ceil_div(heads, PREP_WARPS), PREP_WARPS * 32, 0, st>>>(
                (const double2*)pts_xy, sigma, truncate, meta, n_images, heads, stamps, boxes, wtab, fmask);
        } else {
            dmap_fixed_template_kernel<<<1, 32, 0, st>>>(fixed_sigma, truncate, tmpl, tmpl_tab);
            if (fast)
                dmap_prepare_fast_kernel<<<ceil_div(heads, 256), 256, 0, st>>>((const double2*)pts_xy, meta, n_images, heads, boxes, fmask);
            else
                dmap_prepare_fixed_kernel<<<ceil_div(heads, 256), 256, 0, st>>>((const double2*)pts_xy, tmpl, meta, n_images,
                                                                                heads, stamps, boxes, fmask);
        }
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
        dmap_coarse_kernel<false><<<(unsigned)plan->coarse_tasks, COARSE_THREADS, 0, st>>>(boxes, meta, n_images, ccount,
                                                                                          ctotal, clist);
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
        if (fast)
            dmap_coarse_kernel<true, true><<<(unsigned)plan->coarse_tasks, COARSE_THREADS, 0, st>>>(boxes, meta, n_images, ccount,
                                                                                                   ctotal, clist);
        else
            dmap_coarse_kernel<true><<<(unsigned)plan->coarse_tasks, COARSE_THREADS, 0, st>>>(boxes, meta, n_images, ccount,
                                                                                             ctotal, clist);
        DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    }
    TileDesc* desc = (TileDesc*)(ws + plan->off_desc);
    dmap_tile_setup_kernel<<<ceil_div((int)plan->fine_tiles, 256), 256, 0, st>>>(meta, n_images, (int)plan->fine_tiles, fmask,
                                                                                 ctotal, heads > 0, desc);
    DGVCC_RETURN_IF_CUDA(cudaGetLastError());
    if (fast) {
        static PerDeviceOnce once;
        if (once.first())
            DGVCC_RETURN_IF_CUDA(cudaFuncSetAttribute(dmap_splat_fixed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FAST_SMEM));
        if (heads > 0) dmap_fixed_table_kernel<<<1, 256, 0, st>>>(tmpl_tab, tab2d);
        dmap_splat_fixed_kernel<<<ceil_div((int)plan->fine_tiles, SPLAT_WARPS), SPLAT_THREADS, FAST_SMEM, st>>>(
            desc, (int)plan->fine_tiles, (const unsigned*)clist, tab2d, density);
        return (int)cudaGetLastError();
    }
    // fixed sigma with a narrow stamp: every head shares the template table (wide stamps never use tables)
    dmap_splat_kernel<<<(unsigned)plan->fine_tiles, SPLAT_THREADS, 0, st>>>(stamps, wtab, boxes, desc, clist,
                                                                            sigma ? nullptr : tmpl_tab, density);
    return (int)cudaGetLastError();
}
