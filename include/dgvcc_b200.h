/* dgvcc_b200 -- C ABI of the B200-native density-supervision kernels.
 *
 * The reference (Shimmer93/DGVCC) is pure Python/PyTorch and has no FFI; these
 * entry points are what its three hot-path modules bind through ctypes
 * (INTEGRATION.md shows the stubs).  Each function cites the reference code it
 * replaces.  Conventions (SURVEY.md section 8b):
 *   - every buffer is caller-owned DEVICE memory (torch allocations), passed as
 *     a raw pointer plus sizes; nothing is allocated or freed behind the ABI;
 *   - `stream` is a cudaStream_t (torch.cuda.current_stream().cuda_stream);
 *     launchers never synchronise the host;
 *   - return 0 on success, a negative DGVCC_ERR_* for argument errors, or a
 *     positive cudaError_t; nothing throws across the boundary.
 */
#ifndef DGVCC_B200_H
#define DGVCC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DGVCC_ERR_ARG (-1)
#define DGVCC_ERR_WORKSPACE (-2)
#define DGVCC_ERR_UNSUPPORTED (-3)

/* Element type of the `const void*` feature maps of the *_h entry points. */
#define DGVCC_DTYPE_F16 1
#define DGVCC_DTYPE_BF16 2

/* ABI version; bumped when a signature changes. */
int dgvcc_abi_version(void);

/* 1 when the library was built with -DDGVCC_BOUNDS_CHECK (`DGVCC_BOUNDS_CHECK=1 python -m dgvcc_b200.build`): every
 * kernel then tests the indices it takes from host-built tables and data-dependent computations and traps on a
 * violation (the stand-in for compute-sanitizer, see csrc/common.cuh).  0 for the product build, whose device code
 * does not contain the checks.  No reference counterpart (the reference has no native code). */
int dgvcc_bounds_checked(void);

/* ---------------------------------------------------------------------------
 * Bayesian loss -- replaces losses/bl.py:20-52 (Post_Prob.forward),
 * losses/bl.py:60-80 (Bay_Loss.forward) and the autograd backward of
 * losses/bl.py:88-91 (BL.forward).
 *
 * Ragged inputs are CSR-packed exactly like bl.py:21-22 builds them:
 *   pts_xy      [total_points, 2] f32  (x = column, y = row, image pixels)
 *   targets     [total_points]    f32
 *   meta        int32 host-built table, sections in this order:
 *                 pt_off[B+1]   CSR offsets into pts_xy / targets
 *                 row_off[B+1]  offsets of each image's posterior rows
 *                               (N_i + 1 with background, N_i without, 1 for an
 *                               image with no points: the sum-of-density row)
 *                 keep[B]       ceil(0.9 * (rows_i - 1))  (bl.py:76), host ceil
 *                 icb[B+1]      first point-chunk id of each image
 *                 chunks[C][4]  (image, first point, point count, chunk id to run
 *                               in launch slot c).  Chunks cut every image's points
 *                               into near-equal slices (an image without points has
 *                               one empty chunk) so that all warp tasks cost about the
 *                               same; the last column is a schedule, longest chunks
 *                               first: the sweeps are persistent launches that hand the
 *                               (slot, pixel tile) items out through a work queue.
 *   st_sizes    [B] f32, density [B, hp, wp] f32 (pre_density with the channel
 *   dimension dropped), hp x wp = grid rows x columns, stride = pixels per cell.
 * total_chunks = C; multi_chunk = 1 when some image has more than one chunk.
 * inv_batch = 1 / (global batch size); with image sharding across GPUs every
 * rank passes 1/B_global and all-reduces the returned partial loss.
 * exact_cull != 0 skips (point, pixel-tile) pairs whose exponentials are provably exact zeros
 * (flush-to-zero MUFU.EX2 below 2^-126): bit-identical results, far fewer pairs.  0 = dense.
 * ------------------------------------------------------------------------- */

/* Host-side packing (no CUDA call): the CSR concatenation of bl.py:21-22 plus the int32 table above, written in
 * one pass into the caller's staging buffer (pinned, so that the step uploads ONE buffer).
 *   points[i]  [counts[i], 2] f32 host, targets[i] [counts[i]] f32 host (targets may be NULL: points only);
 *   chunk      points per chunk (big images are cut into near-equal slices of at most this many points);
 *   dst == NULL: only fill `info` (sizes, offsets); otherwise dst must hold info->total_bytes.
 * Layout of dst: table at 0, points at off_points, targets at off_targets (16-byte aligned regions). */
typedef struct dgvcc_bl_packed {
    int64_t total_points, total_rows, total_chunks, multi_chunk;
    int64_t meta_bytes, off_points, off_targets, total_bytes;
} dgvcc_bl_packed;
int dgvcc_bl_pack_host(const float* const* points, const float* const* targets, const int32_t* counts, int batch,
                       int use_background, int chunk, void* dst, size_t dst_bytes, dgvcc_bl_packed* info);

/* Named regions inside the caller-owned workspace (byte offsets), for tests and
 * for the autograd wrapper that keeps the workspace alive until backward. */
typedef struct dgvcc_bl_layout {
    int64_t amax;      /* [B*hp*wp] f32  per-pixel softmax max                       */
    int64_t rz;        /* [B*hp*wp] f32  1 / softmax denominator                     */
    int64_t pbg;       /* [B*hp*wp] f32  posterior of the background row             */
    int64_t ebg;       /* [B*hp*wp] f32  exp(a_bg - amax), un-normalised             */
    int64_t counts;    /* [rows]    f32  expected counts (bl.py:73)                  */
    int64_t wsel;      /* [rows]    f32  sign(c-t) of kept rows, 0 for trimmed rows  */
    int64_t residual;  /* [rows]    f32  |t - c|                                     */
    int64_t loss_img;  /* [B]       f32  per-image trimmed L1                        */
    int64_t ticket;    /* [1]       u32  must be zero on entry (memset once)         */
    int64_t cpart;     /* [tiles*rows] f32 partial counts, one row per CTA of the sweep */
    int64_t zpart;     /* [C*hp*wp] f32  per-chunk share of the softmax denominator  */
    int64_t minpart;   /* (alias of gpart; the per-pixel minima live in the pbg region until it is written) */
    int64_t gpart;     /* [C*hp*wp] f32  per-chunk gradient sums                     */
    int64_t total;     /* bytes needed                                               */
    /* regions of the symmetric (sharded) layout only, 0 otherwise -- dgvcc_bl_shard_workspace_layout */
    int64_t dens;      /* [B*hp*wp] f32  density of the images this rank sweeps      */
    int64_t gfinal;    /* [B*hp*wp] f32  finished gradients, at the image's owner    */
    int64_t flags;     /* [PHASES*world] u32 arrival flags (phase, source rank)      */
    int64_t err;       /* [1] i32        non-zero: a wait timed out (1 + phase + 16*source) */
    int64_t push_ticket; /* [2] u32                                                  */
    int64_t goff;      /* [B*(1024+1)] i32 grid-cell offsets of the points of each image (bl_grid_build_kernel) */
    int64_t gsorted;   /* [rows*2] f32   points sorted by grid cell                   */
    int64_t cshare;    /* [world*share_rows*rows] f32 symmetric layout: the per-CTA partial counts of every rank's band (dgvcc_bl_band_*) */
    int64_t ztick;     /* [B*tiles_img] u32 arrival counters per (image, pixel tile) of bl_z_kernel (zeroed by the forward pass) */
    int64_t gtick;     /* [B*tiles_img] u32 the same for bl_grad_kernel                */
    int64_t queue;     /* [6] u32 work queues of the persistent sweeps (zeroed by the forward pass) */
    int32_t tiles;     /* partial-count rows (CTAs of 4 pixel tiles) per point chunk */
    int32_t rows_per_thread; /* kernel variant chosen for this shape: grid rows ...   */
    int32_t cols_per_thread; /* ... and columns owned by one thread                  */
    int32_t share_rows; /* symmetric layout: partial-count rows reserved per rank in cshare */
} dgvcc_bl_layout;

int dgvcc_bl_workspace_layout(int64_t total_rows, int total_chunks, int batch, int hp, int wp,
                              dgvcc_bl_layout* out);

/* Process-wide tuning knobs for benchmarks and experiments (host side, read when a launch is planned; results do not
 * depend on them beyond the summation order of the expected counts, which follows the pixel tile):
 *   MIN_CELL   smallest cell of the uniform point grid behind the per-pixel minima of bl.py:39, in image pixels
 *              (a power of two, default 64; the cell doubles until the grid has at most 4096 cells)
 *   BAND_TILE  pixel tile per thread of the symmetric (multi-GPU) layouts: 0 = chosen from the task count (default),
 *              82 / 81 / 41 / 21 = rows * 10 + columns.  Must be the same on every rank. */
enum { DGVCC_BL_OPT_MIN_CELL = 0, DGVCC_BL_OPT_BAND_TILE = 1 };
int dgvcc_bl_set_option(int option, int value);

/* Fused forward: per-pixel min / softmax denominator, expected counts, trimmed
 * top-k selection and the loss.  Never materialises the points x pixels matrix.
 * loss_out[0] = inv_batch * sum_i L_i. */
int dgvcc_bl_forward(const float* pts_xy, const float* targets, const int32_t* meta,
                     const float* st_sizes, const float* density,
                     int batch, int hp, int wp, int64_t total_rows, int total_chunks, int multi_chunk,
                     float stride, float sigma, float bg_ratio, int use_bg, int exact_cull, float inv_batch,
                     void* workspace, size_t workspace_bytes, float* loss_out, void* stream);

/* Same launches with caller-created cudaEvent_t handles recorded between them (bench.py's
 * per-kernel timing): events[0] start, [1] after bl_min, [2] after bl_z, [3] after bl_counts,
 * [4] after bl_select.  NULL entries are skipped. */
int dgvcc_bl_forward_profiled(const float* pts_xy, const float* targets, const int32_t* meta,
                              const float* st_sizes, const float* density,
                              int batch, int hp, int wp, int64_t total_rows, int total_chunks, int multi_chunk,
                              float stride, float sigma, float bg_ratio, int use_bg, int exact_cull, float inv_batch,
                              void* workspace, size_t workspace_bytes, float* loss_out, void* stream,
                              void** events);

/* Backward into the density only (bl.py: points carry no grad):
 * grad_density[b,m] = grad_loss[0] * inv_batch * sum_{kept n} sign(c_n - t_n) * p[n,m].
 * Re-uses (and scribbles on the gpart region of) the workspace written by dgvcc_bl_forward. */
int dgvcc_bl_backward(const float* pts_xy, const int32_t* meta,
                      int batch, int hp, int wp, int64_t total_rows, int total_chunks, int multi_chunk,
                      float stride, float sigma, int use_bg, int exact_cull, float inv_batch,
                      const float* grad_loss, void* workspace, size_t workspace_bytes,
                      float* grad_density, void* stream);

/* Materialised posteriors for API parity with Post_Prob.forward (bl.py:20-52):
 * prob_out [total_rows, hp*wp] f32, image i occupying rows row_off[i]..row_off[i+1].
 * (Rows of images without points are filled with 1: the all-background posterior.) */
int dgvcc_bl_posterior(const float* pts_xy, const int32_t* meta, const float* st_sizes,
                       int batch, int hp, int wp, int64_t total_rows, int total_chunks, int multi_chunk,
                       float stride, float sigma, float bg_ratio, int use_bg,
                       void* workspace, size_t workspace_bytes, float* prob_out, void* stream);

/* Bay_Loss.forward on caller-materialised posteriors (bl.py:60-80): expected
 * counts, selection and loss from prob [total_rows, hp*wp]; fills the same
 * workspace regions as dgvcc_bl_forward so dgvcc_bl_bayloss_backward can run.
 * Here the meta table has one (unused) chunk per image: workspace_layout(rows, B, B, ...). */
int dgvcc_bl_bayloss_forward(const float* prob, const float* targets, const int32_t* meta,
                             const float* density, int batch, int hp, int wp, int64_t total_rows,
                             float inv_batch, void* workspace, size_t workspace_bytes,
                             float* loss_out, void* stream);
int dgvcc_bl_bayloss_backward(const float* prob, const int32_t* meta, int batch, int hp, int wp,
                              int64_t total_rows, float inv_batch, const float* grad_loss,
                              const void* workspace, size_t workspace_bytes,
                              float* grad_density, void* stream);

/* ---------------------------------------------------------------------------
 * Bayesian loss, ONE batch spread over the GPUs of a box by point chunks (strong scaling of BASELINE config 3;
 * SURVEY.md 8e).  The reference's unit of independence is the image (losses/bl.py:36,62); an image with 12 000 heads
 * is a quarter of the 16-image batch, so whole-image partitioning stops at 4x on 8 GPUs.  Here the packed point
 * sequence of the batch (bl.py:21-22) is cut into `world` equal contiguous spans; rank r sweeps the chunks of its
 * span over all pixels of the images they belong to, and what an image's other ranks need travels as plain stores
 * into their workspaces over NVLink (peer pointers from dgvcc_peer_open), one arrival flag per (phase, source):
 *   DENS   density of an image, owner -> every rank that sweeps it          (before the expected counts)
 *   Z      per-chunk denominator shares (bl.py:44)                           among the image's ranks
 *          (the minima of bl.py:39 need no exchange: every rank finds them from the replicated points; MIN is unused)
 *   CNT    expected counts + residuals of a rank's rows (bl.py:73-75)        among the image's ranks (top-k needs all)
 *   LOSS   per-image loss, from the rank with the image's first chunk to everybody (summed in image order, bl.py:79)
 *   GPART  per-chunk gradient sums -> the rank with the image's first chunk, which finishes the gradient
 *   GRAD   finished gradient -> the image's owner;  OUT: local gather into the caller's tensor
 * Receivers combine partials in chunk order exactly like dgvcc_bl_forward / _backward, so loss and gradients are
 * bit-identical to the single-GPU call.  No NCCL on the data path.
 * The transfers are fused into the kernels: the sweeps (bl_min / bl_z / bl_grad), the row reduction, the selection
 * and the gradient reduction store their results at home AND on the ranks in the destination mask of the chunk /
 * image as they produce them, and their last CTA raises the flag; the small consumer kernels wait for the flags in
 * their own prologue.  Only DENS (caller's tensor -> workspaces) and OUT are separate copy launches, described by
 * `slices`.  `aux` (DEVICE, uint32): zmask[total_chunks] (ranks that need a chunk's minima / denominator share) |
 * gmask[total_chunks] (rank that finishes the chunk's image, 0 when this rank does) | img_mask[batch] (other ranks
 * of an image) | owner_mask[batch] (owner of an image's gradient, 0 when it is the finishing rank itself).
 *
 * All ranks pass the SAME packed points / targets / st_sizes and the same chunk table (the schedule column lists
 * the rank's own chunk ids in its first chunk_hi - chunk_lo slots); density_local / grad_local hold only the
 * images the rank owns, in the order of the DENS / OUT slices.  `slices` is a DEVICE array, `peers` a DEVICE array of
 * `world` workspace base pointers (own pointer at [rank]); every workspace has dgvcc_bl_shard_workspace_layout.
 * `epoch` must grow by one per forward/backward pair (flags are compared against it); workspaces start zeroed.
 * A wait that sees no flag within 2 s records 1 + phase + 16 * source in the workspace's `err` word and moves on.
 * ------------------------------------------------------------------------- */
#define DGVCC_BL_PHASES 8
enum { DGVCC_BL_PH_DENS = 0, DGVCC_BL_PH_MIN, DGVCC_BL_PH_Z, DGVCC_BL_PH_CNT, DGVCC_BL_PH_LOSS, DGVCC_BL_PH_GPART,
       DGVCC_BL_PH_GRAD, DGVCC_BL_PH_OUT };
typedef struct dgvcc_bl_push {
    int64_t src_off;   /* bytes from the phase's source base (own workspace; density_local for DENS) */
    int64_t dst_off;   /* bytes from the destination rank's workspace (grad_local for OUT)            */
    int32_t bytes;     /* multiple of 4                                                              */
    int32_t dst_rank;
} dgvcc_bl_push;
typedef struct dgvcc_bl_shard {
    int32_t rank, world;
    int32_t chunk_lo, chunk_hi;   /* chunk ids this rank sweeps                         */
    int32_t pt_lo, pt_hi;         /* = packed points [pt_lo, pt_hi)                     */
    int32_t img_lo, img_hi;       /* images it touches                                  */
    int32_t row_lo, row_hi;       /* = posterior rows [row_off[img_lo], row_off[img_hi]) */
    int32_t push_first[DGVCC_BL_PHASES + 1];   /* slices of phase p: [push_first[p], push_first[p+1]) */
    uint32_t wait_mask[DGVCC_BL_PHASES];       /* ranks whose flag of phase p this rank waits for     */
    uint32_t signal_mask[DGVCC_BL_PHASES];     /* ranks this rank signals after its slices of phase p */
    uint32_t epoch;
    int32_t fuse_waits;           /* 1: consumers spin on the flags in their own prologue (one process per GPU);
                                     0: separate one-warp wait kernels (several ranks sharing one GPU / context)   */
    int32_t band_lo, band_hi;     /* dgvcc_bl_band_* only: grid rows [band_lo, band_hi) of EVERY image this rank sweeps */
} dgvcc_bl_shard;
int dgvcc_bl_shard_workspace_layout(int64_t total_rows, int total_chunks, int batch, int hp, int wp, int world,
                                    dgvcc_bl_layout* out);
/* Loads every kernel of the sharded path into the current context (cudaFuncGetAttributes): CUDA loads kernels lazily
 * and a load can wait for running kernels -- such as a peer's wait kernel.  Call once per process / communicator. */
int dgvcc_bl_shard_preload(void);
int dgvcc_bl_shard_forward(const float* pts_xy, const float* targets, const int32_t* meta, const float* st_sizes,
                           const float* density_local, int batch, int hp, int wp, int64_t total_rows, int total_chunks,
                           int multi_chunk, float stride, float sigma, float bg_ratio, int use_bg, int exact_cull,
                           float inv_batch, const dgvcc_bl_shard* shard, const dgvcc_bl_push* slices, const uint32_t* aux,
                           void* const* peers, void* workspace, size_t workspace_bytes, float* loss_out, int defer_loss,
                           void* stream, void** events);
int dgvcc_bl_shard_backward(const float* pts_xy, const int32_t* meta, int batch, int hp, int wp, int64_t total_rows,
                            int total_chunks, float stride, float sigma, int use_bg, int exact_cull, float inv_batch,
                            const float* grad_loss, const dgvcc_bl_shard* shard, const dgvcc_bl_push* slices,
                            const uint32_t* aux, void* const* peers, void* workspace, size_t workspace_bytes,
                            float* grad_local, float* deferred_loss_out, void* stream, void** events);
/* defer_loss != 0: the forward does not wait for the other ranks' per-image losses (a barrier over the whole group that the
 * backward pass does not need); loss_out is then written by dgvcc_bl_shard_backward(deferred_loss_out = the same pointer),
 * i.e. the loss value is complete once the backward launches have run.  The density copy runs on a side stream owned
 * by the library (one per device), forked from and joined to `stream` by events. */
/* `events` (NULL, or caller-created cudaEvent_t handles; NULL entries skipped) are recorded on the stream between the
 * launches, for per-kernel timing.  forward (9): start, after the DENS copy is issued, grid build + minima, bl_z,
 * [wait Z, DENS] finish_z, bl_counts, the row reduction, [wait CNT] selection, [wait LOSS] loss.
 * backward (5): start, bl_grad, [wait GPART] reduction, [wait GRAD] gather, [wait LOSS] deferred loss. */

/* ---------------------------------------------------------------------------
 * Bayesian loss, ONE batch spread over the GPUs of a box by ROW BANDS of the density grid (the strong-scaling path
 * bench.py reports first).  The softmax of bl.py:44 normalises over the points of ONE pixel, so everything per pixel
 * -- the minima of bl.py:39, the denominators, the posteriors, the density gradient -- stays on the rank that owns
 * the pixel; only the expected counts of bl.py:73 sum over pixels.  Rank r sweeps ALL points of every image over the
 * grid rows [band_lo, band_hi) (whole rows of pixel tiles: multiples of dgvcc_bl_layout.rows_per_thread, the last
 * band ends at hp) and the exchange is:
 *   DENS  density rows of an image, owner -> the rank of each band           (side stream, before the counts)
 *   CNT   the per-CTA partial counts of the band (one f32 per posterior row and CTA of pixel tiles), stored by
 *         bl_counts_kernel itself on every rank; all ranks add ALL partial rows in pixel-tile order, so the counts,
 *         the top-k cut (bl.py:76-78) and the loss have the same bits everywhere and no LOSS exchange is needed
 *   GRAD  finished gradient rows, stored by bl_grad_kernel at the image's owner;  OUT: local gather into the caller's tensor
 * One data-dependent exchange in the middle of the step instead of the four of the point-chunk split, and every
 * rank's sweeps are 1/world of the single-GPU sweeps tile for tile.  Results: per-pixel quantities are bit-identical
 * to dgvcc_bl_forward with the same chunk table; so are the counts and the loss whenever the bands are cut at CTA
 * boundaries of the single-GPU sweep (always when 4 divides the column blocks of a tile row, e.g. config 3), else they
 * differ by the order of the partial sums -- identical across ranks and runs, ~1e-7 relative.
 * Arguments as for dgvcc_bl_shard_*: the SAME packed points / targets / table on every rank (every chunk scheduled:
 * the table of dgvcc_bl_pack_host), `shard` with rank / world / band_lo / band_hi / push_first / masks / epoch /
 * fuse_waits (the chunk / point / image / row ranges are ignored), `slices` for DENS and OUT, `owner_mask` (DEVICE,
 * uint32 [batch]): bit of the rank that owns image i, 0 when this rank does.  Workspaces: dgvcc_bl_shard_workspace_layout.
 * events (NULL or cudaEvent_t handles): forward (7) start, DENS issued, grid build + minima, bl_z, [wait DENS]
 * bl_counts (+CNT out), [wait CNT] combine, selection + loss; backward (3) start, bl_grad (+GRAD out), [wait GRAD] gather.
 * The bands are fixed by (hp, rows_per_thread, world): tile rows [n*r/world, n*(r+1)/world) of n = ceil(hp / rows_per_thread).
 * ------------------------------------------------------------------------- */
int dgvcc_bl_band_forward(const float* pts_xy, const float* targets, const int32_t* meta, const float* st_sizes,
                          const float* density_local, int batch, int hp, int wp, int64_t total_rows, int total_chunks,
                          float stride, float sigma, float bg_ratio, int use_bg, int exact_cull, float inv_batch,
                          const dgvcc_bl_shard* shard, const dgvcc_bl_push* slices, const uint32_t* owner_mask,
                          void* const* peers, void* workspace, size_t workspace_bytes, float* loss_out, void* stream,
                          void** events);
int dgvcc_bl_band_backward(const float* pts_xy, const int32_t* meta, int batch, int hp, int wp, int64_t total_rows,
                           int total_chunks, float stride, float sigma, int use_bg, int exact_cull, float inv_batch,
                           const float* grad_loss, const dgvcc_bl_shard* shard, const dgvcc_bl_push* slices,
                           const uint32_t* owner_mask, void* const* peers, void* workspace, size_t workspace_bytes,
                           float* grad_local, void* stream, void** events);

/* Peer-visible device memory for the sharded workspaces (CUDA IPC between the ranks' processes of one box):
 * alloc = cudaMalloc + zero fill; export writes the 64-byte handle a peer process passes to open, which maps the
 * memory into the calling process and enables peer access to the owning GPU. */
int dgvcc_peer_alloc(size_t bytes, void** ptr);
int dgvcc_peer_free(void* ptr);
int dgvcc_peer_export(void* ptr, unsigned char* handle64);
int dgvcc_peer_open(const unsigned char* handle64, void** ptr);
int dgvcc_peer_close(void* ptr);

/* ---------------------------------------------------------------------------
 * Density-map generation -- replaces utils/dmap_gen.py:14-51 (gaussian_filter_density)
 * and utils/dmap_gen.py:53-81 (gaussian_filter_density_fixed).
 *   pts_xy [n,2] f64 (column, row) -- what KDTree(points.copy()) sees, dmap_gen.py:34.
 * ------------------------------------------------------------------------- */

/* KDTree.query(points, k=4) by brute force (dmap_gen.py:34-36) and the adaptive
 * sigma (dmap_gen.py:45-48): nn_idx [n,4] i32 / nn_dist [n,4] f64, column 0 the
 * point itself, missing neighbours (n < 4) = (inf, n) like scipy;
 * sigma[i] = 0.1*(d1+d2+d3) when n > 3, else 15. */
size_t dgvcc_dmap_knn_workspace_bytes(int n);
int dgvcc_dmap_knn_sigma(const double* pts_xy, int n, int32_t* nn_idx, double* nn_dist, double* sigma,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---- batched entry points: a list of images per launch --------------------------------
 * The reference generates one map per call inside a Pool(8) (dmap_gen.py:97-117); here a whole list
 * of images (a single one included) goes through one set of launches.  Heads of all images are packed
 * back to back (pts_xy [total_heads,2] f64, sigma [total_heads] f64), the maps likewise
 * (density: image i occupies [out_off_i, out_off_i + H_i*W_i) floats, row-major [H_i,W_i]).
 *
 * dgvcc_dmap_batch_plan (host only, no CUDA call) fills
 *   meta  [(n_images+1) x DGVCC_DMAP_META_COLS] int64, one row per image + a row of totals:
 *         head offset, heads, H, W, output offset, and the launch bookkeeping of the kernels
 *         (first fine tile / coarse task / coarse-list entry / coarse tile / kNN task / kNN partial);
 *         the caller copies it to the device and passes that DEVICE pointer to the launchers;
 *   plan  totals and the workspace layouts (host struct, passed back by pointer).            */
#define DGVCC_DMAP_META_COLS 12
typedef struct dgvcc_dmap_plan {
    int64_t total_heads, total_pixels, fine_tiles, coarse_tasks, knn_tasks, knn_query_blocks, knn_max_slices;
    int64_t off_stamps, off_boxes, off_wtab, off_fmask, off_tmpl, off_desc, off_ccount, off_ctotal, off_clist, splat_workspace_bytes;
    int64_t off_knn_d2, off_knn_idx, off_knn_pts32, off_knn_max, knn_workspace_bytes;
    int64_t max_side;   /* largest image side of the batch (the fixed-sigma fast path packs pixel indices into 16 bits) */
} dgvcc_dmap_plan;

int dgvcc_dmap_batch_plan(int n_images, const int32_t* heights, const int32_t* widths, const int32_t* counts,
                          int64_t* meta, dgvcc_dmap_plan* plan);

/* dgvcc_dmap_knn_sigma for every image of the batch (neighbours are searched inside each image only).
 * nn_idx [total_heads,4] / nn_dist [total_heads,4] may be NULL when only sigma is wanted. */
int dgvcc_dmap_knn_sigma_batch(const double* pts_xy, int n_images, const int64_t* meta, const dgvcc_dmap_plan* plan,
                               int32_t* nn_idx, double* nn_dist, double* sigma, void* workspace,
                               size_t workspace_bytes, void* stream);

/* density map of every image = sum over its heads, in index order, of
 * scipy.ndimage.gaussian_filter(one_hot, sigma_i, truncate=truncate, mode='constant')
 * (dmap_gen.py:38-49 / 71-79).  sigma == NULL uses fixed_sigma for every head
 * (the fixed variant: sigma 4, truncate 7/4).  Heads with int(y) >= height or
 * int(x) >= width are skipped (dmap_gen.py:41-44) but still count as neighbours.
 * Every pixel of the packed output is written exactly once (zero fill fused):
 * algorithmic HBM traffic 4*H*W + 16*N bytes per image. */
int dgvcc_dmap_splat_batch(const double* pts_xy, const double* sigma, double fixed_sigma, double truncate,
                           int n_images, const int64_t* meta, const dgvcc_dmap_plan* plan, void* workspace,
                           size_t workspace_bytes, float* density, void* stream);

/* ---------------------------------------------------------------------------
 * Dataset-side density handling (SURVEY.md 8f rank 3) -- replaces the density part of
 * DenClsDataset._train_transform (datasets/den_cls_dataset.py:109-150; same block in
 * datasets/den_dataset.py:86-127) and the occupancy map of DenClsDataset.__getitem__
 * (den_cls_dataset.py:60-61) for a whole batch in one launch:
 *   zero padding F.pad(dmap, (left, top, ..)), F.crop(dmap, i, j, crop_h, crop_w),
 *   sum-pool reshape([1, h/d, d, w/d, d]).sum((2, 4)), optional F.hflip, and
 *   bmap = (16 x 16 block sums of the pooled map > 0).
 * maps: packed full-resolution maps f32 (e.g. the output of dgvcc_dmap_splat_batch);
 * meta [batch][DGVCC_DEN_META_COLS] int64 DEVICE table: first float of the map, H, W,
 *   pad_left, pad_top, crop_i (row), crop_j (column), flip (0/1);
 * out_dmap [batch, crop_h/d, crop_w/d] f32; out_bmap [batch, crop_h/d/16, crop_w/d/16] f32
 *   in {0,1}, or NULL (den_dataset.py has no occupancy map).
 * crop_h, crop_w must be multiples of d (the reference's reshape raises otherwise) and,
 * with out_bmap, of 16*d. */
#define DGVCC_DEN_META_COLS 8
int dgvcc_den_train_targets(const float* maps, const int64_t* meta, int batch, int crop_h, int crop_w,
                            int downsample, float* out_dmap, float* out_bmap, void* stream);

/* ---------------------------------------------------------------------------
 * ISW instance-whitening covariance loss -- replaces
 * models/ISW/instance_whitening.py:5-16 (InstanceWhitening = InstanceNorm2d, affine=False),
 * :30-39 (get_covariance_matrix) and :19-27 (instance_whitening_loss) + their autograd.
 *   f_map [batch, c, hw] f32 contiguous (the [B,C,H,W] feature map viewed as [B,C,HW]).
 * ------------------------------------------------------------------------- */

/* y = (x - mean) * invstd per (b,c) plane, biased variance, eps inside the sqrt;
 * planes = B*C.  mean / invstd [planes] are kept for the backward. */
int dgvcc_isw_instnorm_forward(const float* x, int planes, int hw, float eps, float* y, float* mean,
                               float* invstd, void* stream);
int dgvcc_isw_instnorm_backward(const float* dy, const float* y, const float* invstd, int planes, int hw,
                                float* dx, void* stream);

size_t dgvcc_isw_workspace_bytes(int batch, int c, int hw);

/* f_cor [batch,c,c] = bmm(X, X^T) / (hw-1) + 1e-5 * eye  (instance_whitening.py:37).
 * use_tensor_cores != 0 selects the tcgen05/TMA 3xTF32 Gram where the shape tiles
 * (c % 64 == 0, hw % 4 == 0); other shapes use the exact-fp32 CUDA-core Gram. */
int dgvcc_isw_covariance(const float* f_map, const float* eye, int batch, int c, int hw, int use_tensor_cores,
                         void* workspace, size_t workspace_bytes, float* f_cor, void* stream);
/* grad_f_map = (dF + dF^T) X / (hw-1) for an upstream gradient dF of f_cor. */
int dgvcc_isw_covariance_backward(const float* f_map, const float* grad_f_cor, int batch, int c, int hw,
                                  int use_tensor_cores, void* workspace, size_t workspace_bytes, float* grad_f_map,
                                  void* stream);

/* loss[0] = sum_b clamp((sum |f_cor_b * mask| - margin) / num_remove_cov, min=0) / batch
 * (instance_whitening.py:21-25).  margin / num_remove_cov are 1-element DEVICE arrays
 * (the reference passes 0-dim CUDA tensors, cov_settings.py:73). */
int dgvcc_isw_loss_forward(const float* f_cor, const float* mask, const float* margin, const float* num_remove_cov,
                           int batch, int c, int hw, void* workspace, size_t workspace_bytes, float* loss_out,
                           void* stream);
/* grad_f_map for grad_loss[0]; re-uses the workspace written by dgvcc_isw_loss_forward.
 * mask_is_binary != 0 is the caller's promise that every mask entry is 0 or 1 (what CovMatrix_ISW and
 * CovMatrix_IRW produce, cov_settings.py:66-73,103): the upstream matrix is then alpha_b * {0,+-1,+-2}, exact in
 * TF32, and the tensor-core GEMM skips the hi/lo split of that operand.  0 is always correct. */
int dgvcc_isw_loss_backward(const float* f_map, const float* f_cor, const float* mask, const float* num_remove_cov,
                            const float* grad_loss, int batch, int c, int hw, int use_tensor_cores, int mask_is_binary,
                            void* workspace, size_t workspace_bytes, float* grad_f_map, void* stream);

/* cal_covstat (models/ISW/__init__.py:93-104, SURVEY 8f rank 2): var_out [c,c] = unbiased variance over the
 * batch of f_cor * reverse_eye. */
int dgvcc_isw_covstat_var(const float* f_cor, const float* reverse_eye, int batch, int c, float* var_out,
                          void* stream);

/* CovMatrix_ISW.set_mask_matrix (models/ISW/cov_settings.py:52-72), relax_denom != 0 branch:
 * values[i] = (stats[0][i] + stats[1][i] + ...) / count   (the accumulated variance statistics, :84-89, :54)
 * mask[i]   = 1 at the k largest values, else 0; AND-ed with prev_mask when it is not NULL (:70-71).
 * stats [n_stats, n] f32, values / mask / prev_mask [n] f32, n = C*C.  Ties at the k-th value are taken in
 * index order (torch.topk leaves that open).  k = int(num_off_diagonal - margin) is the caller's (:63-65). */
int dgvcc_isw_topk_mask(const float* stats, int n_stats, int count, int n, int k, const float* prev_mask,
                        float* values, float* mask, void* stream);

/* Half-precision feature maps (autocast training): x, y, dy, dx, f_map and grad_f_map are fp16 or bf16 (dtype
 * DGVCC_DTYPE_F16 / DGVCC_DTYPE_BF16, any other value is DGVCC_ERR_ARG); mean, invstd, eye, f_cor and the gradients
 * of f_cor / the loss stay fp32.  Every output is what the fp32 entry points above compute on the map upcast to fp32,
 * rounded to nearest where it is half precision.  The loss forward, the workspace size and the covstat kernel are
 * shared with the fp32 path (they read the fp32 f_cor).
 * The instance norm takes any shape; its backward recomputes y from x, mean and invstd (no saved fp32 y).
 * The Gram and dX = S X run on the tensor cores only: for hw % 8 != 0, c < 32, c % 4 != 0 or a feature-map pointer
 * that is not 16-byte aligned they return DGVCC_ERR_UNSUPPORTED (forward and backward alike), and the caller upcasts. */
int dgvcc_isw_instnorm_forward_h(const void* x, int dtype, int planes, int hw, float eps, void* y, float* mean,
                                 float* invstd, void* stream);
int dgvcc_isw_instnorm_backward_h(const void* dy, const void* x, const float* mean, const float* invstd, int dtype,
                                  int planes, int hw, void* dx, void* stream);
int dgvcc_isw_covariance_h(const void* f_map, int dtype, const float* eye, int batch, int c, int hw, void* workspace,
                           size_t workspace_bytes, float* f_cor, void* stream);
int dgvcc_isw_covariance_backward_h(const void* f_map, int dtype, const float* grad_f_cor, int batch, int c, int hw,
                                    void* workspace, size_t workspace_bytes, void* grad_f_map, void* stream);
int dgvcc_isw_loss_backward_h(const void* f_map, int dtype, const float* f_cor, const float* mask,
                              const float* num_remove_cov, const float* grad_loss, int batch, int c, int hw,
                              int mask_is_binary, void* workspace, size_t workspace_bytes, void* grad_f_map,
                              void* stream);

/* The tensor-core Gram on its own (split-K partial tiles, tests / profiling):
 * part [batch][splits][upper-triangular 128x128 tiles][128][128]. */
int dgvcc_isw_gram_tc_partials(const float* x, int batch, int c, int hw, int splits, int k_per_split,
                               float* part, void* stream);
/* The tensor-core backward GEMM on its own: dx [batch,c,hw] = s [batch,c,c] @ x [batch,c,hw] (3xTF32). */
int dgvcc_isw_sx_tc(const float* s, const float* x, int batch, int c, int hw, float* dx, void* stream);

/* ---------------------------------------------------------------------------
 * Bayesian-dataset target preparation (SURVEY.md section 8f, the step before BL) -- replaces
 * datasets/bay_dataset.py:38-48 (BayesianDataset._cal_dists) and :85-107 (crop block of
 * _train_transform, with utils/misc.py:39-45 cal_inner_area).  is_double selects numpy's dtype
 * rules: 1 for float64 annotations, 0 for float32 ones.
 * ------------------------------------------------------------------------- */

/* dists [n] = mean distance to the 3 nearest heads via sqrt(max(sq_i - 2 p_i.p_j + sq_j, 0)); for
 * n in {2,3} the reference's mean over columns 1.. of the unsorted row.  n < 2 is a no-op (constants). */
int dgvcc_bay_knn_mean(const void* pts_xy, int n, int is_double, void* dists, void* stream);

/* Kept heads (overlap ratio of the clipped box with the crop >= 0.3) in index order:
 * gt_out [kept,2] f64 = (w - (x - left), y - up), targ_out [kept] = ratio, *kept_out = count. */
int dgvcc_bay_crop_targets(const void* gt_xy, const void* dists, int n, int is_double, double crop_left,
                           double crop_up, double crop_right, double crop_down, double* gt_out, void* targ_out,
                           int* kept_out, void* stream);

/* ---------------------------------------------------------------------------
 * Throughput probes used by bench.py for the roofline denominators that
 * MEASURED_PEAKS.json does not carry (SURVEY.md section 8d): chip-wide
 * MUFU.EX2 and FFMA issue rates.  Each launches `iters` dependent-chain rounds
 * on every SM; *ops_out = number of scalar ops the launch executed.
 * ------------------------------------------------------------------------- */
int dgvcc_probe_ex2(float* sink, int iters, int64_t* ops_out, void* stream);
int dgvcc_probe_ffma(float* sink, int iters, int64_t* ops_out, void* stream);
/* mufu_out[i] = ex2.approx.ftz.f32(t[i]) and fma_out[i] = 2^t[i] from the FMA-pipe exponential that the Bayesian-loss
 * sweeps use for an eighth of their pixels (ex2_fma, csrc/common.cuh), for i < n (device arrays): the accuracy check of
 * that function against MUFU.EX2. */
int dgvcc_probe_ex2_fma(const float* t, int n, float* mufu_out, float* fma_out, void* stream);
/* Tensor-pipe probe: every SM issues `iters` x 4 back-to-back tcgen05.mma.kind::tf32 (M=128, N=256, K=8, operands
 * in shared memory, accumulators in TMEM); *flops_out = TF32 flops executed.  The Gram's roofline denominator
 * (SURVEY.md 8d: "Tensor peak for TF32 must also be measured on the box"). */
int dgvcc_probe_tf32(float* sink, int iters, int64_t* flops_out, void* stream);

/* ---------------------------------------------------------------------------
 * Auxiliary Gram-type losses (SURVEY.md 8f rank 4) -- replace losses/lw.py:5-18 (lw_loss) and
 * losses/ortho.py:5-11 (ortho_loss); they reuse the Gram and dX = S X kernels of the ISW path and its
 * workspace (dgvcc_isw_workspace_bytes(batch, c, hw)).
 * ------------------------------------------------------------------------- */

/* lw.py:11-15: yhat = (x - mean) / sqrt(var_unbiased + eps) per (n, c) plane; with a mask [batch, hw]
 * (lw.py:14-15) y_masked = yhat * mask is the Gram input (y_masked may be NULL when mask is NULL).
 * invstd [batch*c] = 1 / sqrt(var + eps), kept for the backward. */
int dgvcc_lw_standardize_forward(const float* x, const float* mask, int batch, int c, int hw, float eps,
                                 float* yhat, float* y_masked, float* invstd, void* stream);
/* dx for an upstream gradient dy of the (masked) standardised map. */
int dgvcc_lw_standardize_backward(const float* dy, const float* yhat, const float* invstd, const float* mask,
                                  int batch, int c, int hw, float* dx, void* stream);

/* gram [batch, c, c] = X X^T (no scaling, no eps): lw.py:16, and the stacked form of ortho.py:9. */
int dgvcc_isw_gram(const float* f_map, int batch, int c, int hw, int use_tensor_cores, void* workspace,
                   size_t workspace_bytes, float* gram, void* stream);

/* lw.py:17-18: loss[0] = sum over samples of sum_{i<j} gram[i][j]^2; backward: grad_y = (dG + dG^T) Y with
 * dG = 2 * grad_loss * triu(gram, 1). */
int dgvcc_lw_loss_forward(const float* gram, int batch, int c, int hw, void* workspace, size_t workspace_bytes,
                          float* loss_out, void* stream);
int dgvcc_lw_loss_backward(const float* y, const float* gram, const float* grad_loss, int batch, int c, int hw,
                           int use_tensor_cores, void* workspace, size_t workspace_bytes, float* grad_y, void* stream);

/* ortho.py:9-11 on the stacked operand z = [x; y] ([2c, p]): gram_zz = dgvcc_isw_gram(z, 1, 2c, p); the block
 * rows 0..c x columns c..2c is x y^T.  loss[0] = mean over c*c of triu(x y^T, 1)^2; backward:
 * grad_x = Sx y, grad_y = Sx^T x with Sx = (2 grad_loss / c^2) triu(x y^T, 1).
 * workspace: dgvcc_isw_workspace_bytes(1, 2c, p). */
int dgvcc_ortho_loss_forward(const float* gram_zz, int c, int p, void* workspace, size_t workspace_bytes,
                             float* loss_out, void* stream);
int dgvcc_ortho_loss_backward(const float* x, const float* y, const float* gram_zz, const float* grad_loss, int c, int p,
                              int use_tensor_cores, void* workspace, size_t workspace_bytes, float* grad_x,
                              float* grad_y, void* stream);

/* Half-precision inputs of the auxiliary losses (autocast training; dtype DGVCC_DTYPE_F16 / DGVCC_DTYPE_BF16): every
 * output is what the fp32 entry points above compute on the input upcast to fp32, bit for bit, gradients rounded to
 * nearest into the input type.  The Gram and dX = S X run on the tensor cores only: for hw (p) % 8 != 0, c < 32,
 * c % 4 != 0 or a half-precision pointer that is not 16-byte aligned they return DGVCC_ERR_UNSUPPORTED, and the caller
 * upcasts.  mean, sd, invstd [batch*c], mask [batch, hw] (or NULL), gram and grad_y stay fp32. */
/* lw.py:16 and ortho.py:9 on a half map: gram [batch, c, c] = X X^T, as dgvcc_isw_gram. */
int dgvcc_isw_gram_h(const void* f_map, int dtype, int batch, int c, int hw, void* workspace, size_t workspace_bytes,
                     float* gram, void* stream);
/* ortho.py:9-11 backward on half x, y [c, p]; grad_x, grad_y half. */
int dgvcc_ortho_loss_backward_h(const void* x, const void* y, int dtype, const float* gram_zz, const float* grad_loss,
                                int c, int p, void* workspace, size_t workspace_bytes, void* grad_x, void* grad_y,
                                void* stream);
/* lw.py:11-13: the statistics of dgvcc_lw_standardize_forward only (mean, sd = sqrt(var + eps), invstd = 1 / sd); the
 * standardised map is never written. */
int dgvcc_lw_standardize_stats_h(const void* x, int dtype, int batch, int c, int hw, float eps, float* mean, float* sd,
                                 float* invstd, void* stream);
/* lw.py:13-16: gram = Y Y^T with Y = (x - mean) / sd (* mask) standardised inside the Gram kernel. */
int dgvcc_lw_gram_h(const void* x, int dtype, const float* mean, const float* sd, const float* mask, int batch, int c,
                    int hw, void* workspace, size_t workspace_bytes, float* gram, void* stream);
/* Backward of lw.py:16-18: grad_y [batch, c, hw] fp32 = (dG + dG^T) Y, Y standardised inside the GEMM, as
 * dgvcc_lw_loss_backward on Y. */
int dgvcc_lw_loss_backward_h(const void* x, int dtype, const float* mean, const float* sd, const float* mask,
                             const float* gram, const float* grad_loss, int batch, int c, int hw, void* workspace,
                             size_t workspace_bytes, float* grad_y, void* stream);
/* Backward of lw.py:11-15: dx (half) from dy (fp32); yhat is recomputed from x, mean and sd. */
int dgvcc_lw_standardize_backward_h(const float* dy, const void* x, int dtype, const float* mean, const float* sd,
                                    const float* invstd, const float* mask, int batch, int c, int hw, void* dx,
                                    void* stream);

/* ---------------------------------------------------------------------------
 * Switchable whitening (SURVEY.md 8f rank 4) -- replaces SwitchWhiten2d.forward
 * (models/ISW/switchwhiten.py:84-183) and SyncMeanCov / SyncSwitchWhiten2d.forward
 * (models/ISW/sync_switchwhiten.py:9-56,135-223) with hand-derived backward passes.
 *
 * x, y, grad_y, grad_x: fp32 [n, channels, hw] contiguous; groups = channels / num_pergroup, num_pergroup in
 * {4, 8, 16}; sw_type in {2, 3, 5}; 1 <= T <= 8.  Statistics are fp64 device arrays owned by the caller:
 *   mean_in [n, channels]   cov_in [n, groups, cp, cp]   mean_bn [channels]   cov_bn [groups, cp, cp]
 * The four exchanges of SyncMeanCov happen BETWEEN these calls, on mean_bn / cov_bn / grad_mean_bn / grad_cov_bn
 * (sum over ranks, then the caller divides the forward ones by the world size).
 * ------------------------------------------------------------------------- */

#define DGVCC_SW_MAX_T 8

/* Bytes of the scratch workspace shared by every call below for one layer invocation (the backward calls keep
 * intermediate adjoints in it between dgvcc_sw_backward_stats and dgvcc_sw_backward_apply).  0 on bad arguments. */
size_t dgvcc_sw_workspace_bytes(int n, int channels, int hw, int num_pergroup);

/* One read of x: per-sample channel means and group covariances, centred, divided by hw
 * (switchwhiten.py:117-121). */
int dgvcc_sw_instance_stats(const float* x, int n, int channels, int hw, int num_pergroup, double* mean_in,
                            double* cov_in, void* workspace, size_t workspace_bytes, void* stream);

/* This rank's batch mean (switchwhiten.py:94 / sync_switchwhiten.py:19) and, given the (exchanged) mean, this rank's
 * batch covariance centred on it (switchwhiten.py:95-98 / sync_switchwhiten.py:22-23), both from the per-sample
 * statistics: cov_bn = mean_n(cov_in + d d^T), d = mean_in - mean_bn. */
int dgvcc_sw_batch_mean(const double* mean_in, int n, int channels, double* mean_bn, void* stream);
int dgvcc_sw_batch_cov(const double* mean_in, const double* cov_in, const double* mean_bn, int n, int channels,
                       int num_pergroup, double* cov_bn, void* stream);

/* switchwhiten.py:101-104 / sync_switchwhiten.py:28-31 on fp32 buffers running_mean [channels], running_cov
 * [groups, cp, cp]: running = running * momentum + one_minus_momentum * batch, rounded like the four torch ops
 * (the caller passes 1 - momentum as its host language computes it). */
int dgvcc_sw_update_running(float* running_mean, float* running_cov, const double* mean_bn, const double* cov_bn,
                            int channels, int num_pergroup, double momentum, double one_minus_momentum, void* stream);

/* Mixes the statistics with softmax(sw_mean_weight), softmax(sw_var_weight) (sw_var_weight NULL = tie_weight),
 * runs T Newton iterations per (sample, group) (switchwhiten.py:166-175) and applies
 * y = weight * (wm (x - mean)) + bias (weight / bias NULL = affine=False) in one pass over x.
 * a_fwd [n, groups, cp, cp] fp32 = diag(weight) wm is kept for the backward. */
int dgvcc_sw_whiten_forward(const float* x, const double* mean_in, const double* cov_in, const double* mean_bn,
                            const double* cov_bn, const float* sw_mean_weight, const float* sw_var_weight,
                            const float* weight, const float* bias, int n, int channels, int hw, int num_pergroup,
                            int sw_type, int T, float eps, float* a_fwd, float* y, void* workspace,
                            size_t workspace_bytes, void* stream);

/* Backward, first half: one read of x and grad_y, the adjoint of the Newton iteration per (sample, group), and the
 * reductions over samples.  Outputs: grad_sw_mean [sw_type], grad_sw_var [sw_type] (NULL when tied: the sum goes to
 * grad_sw_mean), grad_weight / grad_bias [channels] (NULL = affine=False), and this rank's adjoints of the batch
 * statistics grad_mean_bn [channels], grad_cov_bn [groups, cp, cp] (fp64) -- the two backward exchanges of
 * sync_switchwhiten.py:44-45 act on them. */
int dgvcc_sw_backward_stats(const float* x, const float* grad_y, const double* mean_in, const double* cov_in,
                            const double* mean_bn, const double* cov_bn, const float* sw_mean_weight,
                            const float* sw_var_weight, const float* weight, int n, int channels, int hw,
                            int num_pergroup, int sw_type, int T, float eps, float* grad_sw_mean, float* grad_sw_var,
                            float* grad_weight, float* grad_bias, double* grad_mean_bn, double* grad_cov_bn,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Backward, second half: grad_x = a_fwd^T grad_y + M2 x + const in one pass over x and grad_y.
 * bn_scale = 1 / (n * hw * world_size) when the batch statistics were computed from x (training), 1 / (n * hw) for
 * the synchronised layer in eval mode (sync_switchwhiten.py:48-55 back-propagates through the running statistics),
 * 0 for the plain layer in eval mode. */
int dgvcc_sw_backward_apply(const float* x, const float* grad_y, const float* a_fwd, const double* mean_in,
                            const double* mean_bn, const double* grad_mean_bn, const double* grad_cov_bn,
                            const float* sw_mean_weight, const float* sw_var_weight, double bn_scale, int n,
                            int channels, int hw, int num_pergroup, int sw_type, float* grad_x, void* workspace,
                            size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DGVCC_B200_H */
