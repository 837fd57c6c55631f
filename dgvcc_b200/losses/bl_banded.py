"""Bayesian loss of ONE batch spread over the GPUs of a box by ROW BANDS of the density grid (strong scaling; SURVEY.md 8e).

The softmax of the reference (losses/bl.py:44) normalises over the points of ONE pixel.  Splitting the batch by
pixels therefore keeps the per-pixel minima (bl.py:39), denominators, posteriors and the density gradient on the rank
that owns the pixel; only the expected counts (bl.py:73: a sum over pixels) cross ranks.  Rank r sweeps ALL points of
every image over the grid rows ``[band_lo[r], band_hi[r])`` -- the single-GPU sweeps restricted to 1/world of their
pixel tiles -- and the step has ONE data-dependent exchange (include/dgvcc_b200.h, ``dgvcc_bl_band_*``):

    DENS  density rows, owner -> band ranks (side stream)      CNT  per-CTA partial counts -> everybody (added in tile order)
    GRAD  finished gradient rows, band rank -> owner           (no LOSS exchange: every rank finds the same loss)

against four dependent exchanges for the point-chunk split of ``bl_sharded.ChunkShardedBL`` (kept: it needs no
replicated sweep over the points of an image, which matters only when a rank cannot hold the whole batch's points --
never the case for this loss: 50 000 heads are 400 KB).

    comm = IpcComm()                                   # one per process, after init_process_group
    loss_fn = BandShardedBL(sigma, c_size, stride, background_ratio, use_background, device, comm)
    loss = loss_fn(points, st_sizes, targets, pre_density_local, owners)      # the same bits on every rank
    loss.backward()                                    # pre_density_local.grad: the maps this rank owns

Interface and communicators as in ``bl_sharded`` (``LocalComm`` runs the ranks inside one process on one GPU).
"""
import ctypes

import numpy as np

from .. import _native
from . import bl as _bl
from .bl_sharded import IpcComm, LocalComm, _cached_plan, _PeerBL, _PeerPlan  # noqa: F401  (IpcComm, LocalComm: re-exported)

FORCE_CHUNK = None   # experiments: points per chunk of the band plan, whatever the world size
TAIL_SPLIT = 0       # experiments: cut the last quarter of every image's chunks into this many pieces (build_meta)


def band_chunk_points(total_points, world, hp, wp):
    """Points per chunk when every rank sweeps 1/world of the pixel tiles.  A rank should see about 1.7 rounds of warp
    tasks (8 x 32 pixel tiles; 16 resident warps on each of 148 SMs): fewer, and the tail of a sweep is one full-length
    task; more, and the per-task prologues, the per-chunk partial arrays and the last arrival's sum over the chunks of a
    tile grow.  Measured on 8 B200 with BASELINE config 3 (profiles/r2_strong_scaling.md; step time against points per
    chunk): 192 -> 0.4225 ms, 256 -> 0.4268, 320 -> 0.4215, 384 -> 0.4295, 512 -> 0.4442; on 2 B200 256 and 512 are within
    1 %.  Between 256 and the single-GPU chunk size, a multiple of 32."""
    if FORCE_CHUNK:
        return int(FORCE_CHUNK)
    tiles = -(-wp // 32) * -(-hp // 8)
    want_chunks = -(-148 * 16 * 5 * max(world, 1) // (3 * max(tiles, 1)))
    want = -(-max(total_points, 1) // want_chunks)
    return int(min(_bl.chunk_points(), max(256, -(-want // 32) * 32)))


class BandPlan(_PeerPlan):
    """What the ranks agree on, from the head counts and the grid shape alone (host, deterministic)."""

    def __init__(self, counts, use_bg, world, owners, hp, wp, chunk):
        super().__init__(counts, use_bg, world, owners, hp, wp)
        self.chunk = int(chunk)
        self.meta, self.total_chunks, self.multi_chunk = _bl.build_meta(self.counts, self.rows, self.chunk, TAIL_SPLIT)
        self._query_layout()
        # bands: whole rows of pixel tiles (rows_per_thread grid rows each), as equal as they come
        tile_rows = self.layout.rows_per_thread
        n_tr = -(-hp // tile_rows)
        cut = (np.arange(world + 1, dtype=np.int64) * n_tr) // world
        self.band_lo = np.minimum(cut[:-1] * tile_rows, hp)
        self.band_hi = np.minimum(cut[1:] * tile_rows, hp)
        self._build_tables()
        for r, sh in enumerate(self.shards):
            sh.band_lo, sh.band_hi = int(self.band_lo[r]), int(self.band_hi[r])

    def meta_for(self, rank):
        """The int32 table of include/dgvcc_b200.h: the same on every rank, every chunk scheduled."""
        return self.meta

    def _exchange(self, flag, add):
        w, L, b = self.world, self.layout, self.batch
        m4, row4 = 4 * self.hp * self.wp, 4 * self.wp
        P = _native
        owner_mask = np.zeros((w, b), dtype=np.uint32)
        for i in range(b):
            own = int(self.owners[i])
            k_local = int(np.searchsorted(self.owned[own], i))
            for q in range(w):
                lo, hi = int(self.band_lo[q]), int(self.band_hi[q])
                if hi > lo:   # density rows of the band: owner -> band rank (the owner's own band included)
                    add(P.BL_PH_DENS, own, k_local * m4 + lo * row4, q, L.dens + i * m4 + lo * row4, (hi - lo) * row4)
                    flag(P.BL_PH_DENS, own, q)
                if q != own:  # finished gradient rows: every rank -> owner (ranks without a band just raise the flag)
                    owner_mask[q, i] = np.uint32(1 << own)
                flag(P.BL_PH_GRAD, q, own)
            add(P.BL_PH_OUT, own, L.gfinal + i * m4, own, k_local * m4, m4)
        for r in range(w):        # count shares: everybody -> everybody
            for q in range(w):
                flag(P.BL_PH_CNT, r, q)
        return [owner_mask[r].copy() for r in range(w)]


_plan_cache = {}


def plan_bands(counts, use_bg, world, owners, hp, wp, chunk=None):
    """Cached ``BandPlan`` (forward and backward of one step share it; a benchmark hits it every step)."""
    key = (tuple(int(c) for c in counts), bool(use_bg), int(world), None if owners is None else tuple(int(o) for o in owners),
           int(hp), int(wp), int(chunk or band_chunk_points(sum(int(c) for c in counts), world, hp, wp)), int(TAIL_SPLIT))
    return _cached_plan(_plan_cache, key, lambda: BandPlan(counts, use_bg, world, owners, hp, wp, key[-2]))


class BandShardedBL(_PeerBL):
    """``BL`` for one batch spread over ``comm.world`` GPUs by row bands of the density grid (module docstring)."""

    FWD_PHASES = ["issue DENS copy (side stream)", "grid build + minima", "z (+ finish)", "[wait DENS] counts (+CNT out)",
                  "[wait CNT] combine", "select + loss"]
    BWD_PHASES = ["grad (+ finish, GRAD out)", "[wait GRAD] gather"]

    def __init__(self, sigma, c_size, stride, background_ratio, use_background, device, comm):
        super().__init__(sigma, c_size, stride, background_ratio, use_background, device, comm)
        self.chunk = None    # points per chunk (None: band_chunk_points)

    def _plan(self, counts, owners, hp, wp):
        return plan_bands(counts, self.post_prob.use_bg, self.comm.world, owners, hp, wp, self.chunk)

    def _forward(self, plan, packed, st, dens, inv_batch, shard, tables, loss, backward_follows):
        """dgvcc_bl_band_forward: the loss is complete when it returns (every rank finds it for itself)."""
        comm, pp = self.comm, self.post_prob
        rc = _native.lib().dgvcc_bl_band_forward(
            _native.ptr(packed.pts), _native.ptr(packed.targets), _native.ptr(packed.meta), _native.ptr(st), _native.ptr(dens),
            plan.batch, plan.hp, plan.wp, plan.total_rows, plan.total_chunks, float(pp.stride), float(pp.sigma),
            float(pp.bg_ratio), int(pp.use_bg), int(self.exact_cull), inv_batch, ctypes.byref(shard), _native.ptr(tables[0]),
            _native.ptr(tables[1]), _native.ptr(comm.peer_table), _native.ptr(comm.workspace), comm.nbytes, _native.ptr(loss),
            _native.stream_ptr(comm.device), self._event_handles("fwd"))
        _native.check(rc, "dgvcc_bl_band_forward")
        return None

    def _backward(self, plan, packed, inv_batch, g, shard, tables, grad, deferred):
        comm, pp = self.comm, self.post_prob
        rc = _native.lib().dgvcc_bl_band_backward(
            _native.ptr(packed.pts), _native.ptr(packed.meta), plan.batch, plan.hp, plan.wp, plan.total_rows,
            plan.total_chunks, float(pp.stride), float(pp.sigma), int(pp.use_bg), int(self.exact_cull), inv_batch,
            _native.ptr(g), ctypes.byref(shard), _native.ptr(tables[0]), _native.ptr(tables[1]), _native.ptr(comm.peer_table),
            _native.ptr(comm.workspace), comm.nbytes, _native.ptr(grad), _native.stream_ptr(comm.device),
            self._event_handles("bwd"))
        _native.check(rc, "dgvcc_bl_band_backward")
