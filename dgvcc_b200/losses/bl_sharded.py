"""Bayesian loss of ONE batch spread over the GPUs of a box by point chunks (strong scaling; SURVEY.md 8e).

The reference's independent unit is the image (losses/bl.py:36,62-79).  One QNRF image with 12 000 heads is a
quarter of BASELINE config 3's 16-image batch, so assigning whole images to ranks stops at ~4x on 8 GPUs.  Here
the packed point sequence of the batch (the concatenation of bl.py:21-22) is cut into ``world`` equal spans;
rank r sweeps the chunks of its span, and the partial results an image's other ranks need are written straight
into their workspaces over NVLink (csrc/bl_kernels.cu, "point-chunk sharding"; include/dgvcc_b200.h lists the
exchange phases).  Partials are combined in chunk order exactly like on one GPU: loss and gradients are
bit-identical to ``BL`` on a single device.

    comm = IpcComm()                                   # one per process, after init_process_group
    loss_fn = ChunkShardedBL(sigma, c_size, stride, background_ratio, use_background, device, comm)
    loss = loss_fn(points, st_sizes, targets, pre_density_local, owners)      # the same value on every rank
    loss.backward()                                    # pre_density_local.grad: the maps this rank owns

``points`` / ``targets`` / ``st_sizes`` describe the WHOLE batch and are the same on every rank (a few hundred KB);
``pre_density_local`` holds the predicted maps of the images this rank owns (``owners[i]`` = rank of image i, default:
contiguous blocks, what a data-parallel model produces), in image order.

``plan_shards`` (host only, numpy) is the whole bookkeeping: chunk table, per-rank ranges, push slices, wait /
signal masks.  ``LocalComm`` runs several "ranks" inside one process on one GPU (one stream each) -- the parity
tests use it, the kernels and the protocol are the same as with one process per GPU.

The row-band split (``bl_banded``) shares this module's communicators and host layer: the plan base ``_PeerPlan``
(owners, workspace layout, exchange tables), the module base ``_PeerBL`` and the autograd function ``_PeerFn``.
"""
import ctypes

import numpy as np
import torch
from torch.nn import Module

from .. import _native
from . import bl as _bl

SLICE_BYTES = 32 * 1024   # one CTA of the push kernel moves at most this much


class _PeerPlan:
    """What the ranks of either peer split agree on, computed from the head counts alone (host, deterministic): the
    owners of the images' density, the posterior rows, the symmetric workspace layout and the exchange tables.  A
    split's constructor adds its partition, then calls ``_query_layout`` and ``_build_tables``."""

    def __init__(self, counts, use_bg, world, owners, hp, wp):
        counts = np.asarray(counts, dtype=np.int64)
        b = len(counts)
        if b == 0:
            raise ValueError("empty batch")
        self.batch, self.world, self.use_bg, self.hp, self.wp = b, int(world), bool(use_bg), int(hp), int(wp)
        owners = np.asarray(owners if owners is not None else np.arange(b) * world // b, dtype=np.int64)
        if owners.shape != (b,) or owners.min() < 0 or owners.max() >= world:
            raise ValueError("owners must give one rank in [0, world) per image")
        self.owners, self.counts = owners, counts
        self.rows = np.where(counts == 0, 1, counts + (1 if use_bg else 0))
        self.total_points, self.total_rows = int(counts.sum()), int(self.rows.sum())
        self.owned = [np.nonzero(owners == r)[0] for r in range(world)]          # images whose density lives on rank r

    def _query_layout(self):
        self.layout = _native.BLLayout()
        _native.check(_native.lib().dgvcc_bl_shard_workspace_layout(self.total_rows, self.total_chunks, self.batch, self.hp,
                                                                    self.wp, self.world, self.layout),
                      "dgvcc_bl_shard_workspace_layout")

    def _build_tables(self):
        """Who sends what to whom.  DENS and OUT are copy launches described by slices; the other phases are fused into
        the kernels, which only need destination masks (``aux``) -- and every phase needs its wait / signal masks.  The
        split's ``_exchange(flag, add)`` names the transfers and returns the ``aux`` array of every rank; the split
        fills its own ``BLShard`` fields afterwards."""
        w, n_ph = self.world, _native.BL_PHASES
        per = [[[] for _ in range(n_ph)] for _ in range(w)]        # per[src][phase] = [(src_off, dst_off, bytes, dst)]
        wait = np.zeros((w, n_ph), dtype=np.uint32)
        signal = np.zeros((w, n_ph), dtype=np.uint32)

        def flag(phase, src, dst):
            if dst != src:
                wait[dst, phase] |= np.uint32(1 << src)
                signal[src, phase] |= np.uint32(1 << dst)

        def add(phase, src, src_off, dst, dst_off, nbytes):
            step = SLICE_BYTES if (src_off | dst_off | nbytes) % 16 == 0 else 1 << 30
            for o in range(0, nbytes, step):
                per[src][phase].append((src_off + o, dst_off + o, min(step, nbytes - o), dst))

        self.aux = self._exchange(flag, add)
        self.slices, self.shards, self._dev = [], [], {}
        for r in range(w):
            rows, first = [], [0]
            for ph in range(n_ph):
                rows += per[r][ph]
                first.append(len(rows))
            arr = np.zeros((max(len(rows), 1), 3), dtype=np.int64)   # (src_off, dst_off, bytes | dst_rank << 32): 24-byte records
            if rows:
                t = np.asarray(rows, dtype=np.int64)
                arr[:len(rows), 0], arr[:len(rows), 1] = t[:, 0], t[:, 1]
                arr[:len(rows), 2] = t[:, 2] | (t[:, 3] << 32)
            self.slices.append(arr)
            sh = _native.BLShard()
            sh.rank, sh.world = r, w
            for ph in range(n_ph + 1):
                sh.push_first[ph] = first[ph]
            for ph in range(n_ph):
                sh.wait_mask[ph], sh.signal_mask[ph] = int(wait[r, ph]), int(signal[r, ph])
            self.shards.append(sh)

    def tables_on(self, rank, device):
        """(slices, aux) of ``rank`` as device tensors (uploaded once per plan)."""
        key = (rank, str(device))
        t = self._dev.get(key)
        if t is None:
            t = self._dev[key] = (torch.from_numpy(self.slices[rank]).to(device),
                                  torch.from_numpy(self.aux[rank].view(np.int32)).to(device))
        return t


def _cached_plan(cache, key, make):
    """``cache[key]``, made by ``make()`` when missing (a cache of more than 64 plans is emptied first)."""
    plan = cache.get(key)
    if plan is None:
        if len(cache) > 64:
            cache.clear()
        plan = cache[key] = make()
    return plan


class ShardPlan(_PeerPlan):
    """The plan of the point-chunk split: chunk table, per-rank point spans, and the exchange of every phase."""

    def __init__(self, counts, use_bg, world, owners, hp, wp, chunk):
        super().__init__(counts, use_bg, world, owners, hp, wp)
        b, counts = self.batch, self.counts
        pt_off = np.concatenate(([0], np.cumsum(counts)))
        row_off = np.concatenate(([0], np.cumsum(self.rows)))
        self.pt_off, self.row_off = pt_off, row_off
        total = self.total_points
        bounds = (np.arange(world + 1, dtype=np.int64) * total) // world   # rank r sweeps points [bounds[r], bounds[r+1])
        self.bounds = bounds
        rank_of = lambda pos: min(int(np.searchsorted(bounds[1:], pos, side="right")), world - 1)  # noqa: E731

        img, start, cnt, owner = [], [], [], []
        for i in range(b):
            lo, hi = int(pt_off[i]), int(pt_off[i + 1])
            if hi == lo:   # an image without points still has its sum-of-density row (bl.py:63-65): one empty chunk
                img.append(i); start.append(0); cnt.append(0); owner.append(rank_of(lo))
                continue
            for r in range(rank_of(lo), rank_of(hi - 1) + 1):
                a, e = max(lo, int(bounds[r])), min(hi, int(bounds[r + 1]))
                if e <= a:
                    continue
                n_sub = -(-(e - a) // chunk)
                for k in range(n_sub):
                    s0, s1 = a + (e - a) * k // n_sub, a + (e - a) * (k + 1) // n_sub
                    img.append(i); start.append(s0 - lo); cnt.append(s1 - s0); owner.append(r)
        self.c_img, self.c_start, self.c_cnt, self.c_owner = (np.asarray(v, dtype=np.int64) for v in (img, start, cnt, owner))
        self.total_chunks = len(img)
        assert (np.diff(self.c_owner) >= 0).all() and (np.diff(self.c_img) >= 0).all()
        self.icb = np.searchsorted(self.c_img, np.arange(b + 1), side="left")   # first chunk of each image
        self.multi_chunk = int((np.diff(self.icb) > 1).any())
        self.chunk_lo = np.searchsorted(self.c_owner, np.arange(world), side="left")
        self.chunk_hi = np.searchsorted(self.c_owner, np.arange(world), side="right")
        self.lead = self.c_owner[self.icb[:-1]]                                  # rank with the image's first chunk
        self.groups = [sorted(set(self.c_owner[self.icb[i]:self.icb[i + 1]].tolist())) for i in range(b)]
        self.img_lo = np.array([self.c_img[self.chunk_lo[r]] if self.chunk_hi[r] > self.chunk_lo[r] else 0 for r in range(world)])
        self.img_hi = np.array([self.c_img[self.chunk_hi[r] - 1] + 1 if self.chunk_hi[r] > self.chunk_lo[r] else 0
                                for r in range(world)])
        self._query_layout()
        self._build_tables()
        for r, sh in enumerate(self.shards):
            sh.chunk_lo, sh.chunk_hi = int(self.chunk_lo[r]), int(self.chunk_hi[r])
            sh.pt_lo, sh.pt_hi = int(self.bounds[r]), int(self.bounds[r + 1])
            sh.img_lo, sh.img_hi = int(self.img_lo[r]), int(self.img_hi[r])
            sh.row_lo, sh.row_hi = int(self.row_off[sh.img_lo]), int(self.row_off[sh.img_hi])

    # ------------------------------------------------------------------------------------------------ meta table
    def meta_for(self, rank):
        """The int32 table of include/dgvcc_b200.h; the schedule column lists this rank's own chunks first."""
        b, c = self.batch, self.total_chunks
        meta = np.zeros(4 * b + 3 + 4 * c, dtype=np.int32)
        meta[:b + 1] = self.pt_off
        meta[b + 1:2 * b + 2] = self.row_off
        meta[2 * b + 2:3 * b + 2] = np.ceil(0.9 * (self.rows - 1).astype(np.float64))   # bl.py:76
        meta[3 * b + 2:4 * b + 3] = self.icb
        table = meta[4 * b + 3:].reshape(c, 4)
        table[:, 0], table[:, 1], table[:, 2] = self.c_img, self.c_start, self.c_cnt
        mine = np.arange(self.chunk_lo[rank], self.chunk_hi[rank]) if rank is not None else np.arange(c)
        order = mine[np.argsort(-self.counts[self.c_img[mine]], kind="stable")]       # chunks of the big images first
        table[:len(order), 3] = order
        return meta

    def meta_all(self):
        """The same chunk table with every chunk scheduled: what ONE GPU runs through dgvcc_bl_forward / _backward to
        produce the bits the sharded ranks must reproduce (tests)."""
        return self.meta_for(None)

    # ------------------------------------------------------------------------------------------------ exchange plan
    def _exchange(self, flag, add):
        w, L, m4 = self.world, self.layout, 4 * self.hp * self.wp
        P = _native
        c, b = self.total_chunks, self.batch
        zmask = np.zeros((w, c), dtype=np.uint32)      # per rank: destinations of a chunk's minima / denominator share
        gmask = np.zeros((w, c), dtype=np.uint32)      # rank that finishes the chunk's image (0: this rank itself)
        img_mask = np.zeros((w, b), dtype=np.uint32)   # the image's other ranks
        owner_mask = np.zeros((w, b), dtype=np.uint32)  # owner of the image's gradient (0: the finishing rank itself)
        for i in range(b):
            g, lead, own = self.groups[i], int(self.lead[i]), int(self.owners[i])
            k_local = int(np.searchsorted(self.owned[own], i))
            for q in g:                                   # density: owner -> every rank that sweeps the image
                add(P.BL_PH_DENS, own, k_local * m4, q, L.dens + i * m4, m4)
                flag(P.BL_PH_DENS, own, q)
            c0, c1 = int(self.icb[i]), int(self.icb[i + 1])
            for ch in range(c0, c1):
                r = int(self.c_owner[ch])
                for q in g:
                    if q != r:                            # denominator shares: among the image's ranks
                        zmask[r, ch] |= np.uint32(1 << q)
                        flag(P.BL_PH_Z, r, q)
                if r != lead:                             # gradient sums -> the rank with the image's first chunk
                    gmask[r, ch] = np.uint32(1 << lead)
                    flag(P.BL_PH_GPART, r, lead)
            for r in g:                                   # expected counts + residuals of a rank's rows: among the image's ranks
                for q in g:
                    if q != r:
                        img_mask[r, i] |= np.uint32(1 << q)
                        flag(P.BL_PH_CNT, r, q)
            for q in range(w):                            # the image's loss: lead -> everybody
                flag(P.BL_PH_LOSS, lead, q)
            if own != lead:                               # finished gradient -> owner
                owner_mask[lead, i] = np.uint32(1 << own)
                flag(P.BL_PH_GRAD, lead, own)
            add(P.BL_PH_OUT, own, L.gfinal + i * m4, own, k_local * m4, m4)
        return [np.concatenate([zmask[r], gmask[r], img_mask[r], owner_mask[r]]).astype(np.uint32) for r in range(w)]


_plan_cache = {}


FORCE_CHUNK = None   # experiments: points per chunk of the sharded plan, whatever the world size


def shard_chunk_points(total_points, world):
    """Points per chunk for a batch spread over ``world`` ranks: about 18 chunks per rank (and per 18 x 1024 points).
    Measured on 8 B200 with BASELINE config 3 (profiles/r2_strong_scaling.md; step time against points per chunk):
    128 -> 0.50 ms, 192 -> 0.46, 256 -> 0.48, 352 -> 0.447, 448 -> 0.45, 704 -> 0.50.  Small chunks pay the per-task
    prologues / epilogues and per-chunk partial arrays, large ones leave a rank with too few CTAs to fill its SMs.
    Never above the single-GPU chunk size, never below 128, a multiple of 32."""
    if FORCE_CHUNK:
        return int(FORCE_CHUNK)
    per_rank = max(1, -(-total_points // max(world, 1)))
    waves = max(1, -(-per_rank // (18 * _bl.chunk_points())))
    want = -(-per_rank // (18 * waves))
    return int(min(_bl.chunk_points(), max(128, -(-want // 32) * 32)))


def plan_shards(counts, use_bg, world, owners, hp, wp, chunk=None):
    """Cached ``ShardPlan`` (a training loop sees few distinct count tuples per epoch only in benchmarks, but the
    plan of the previous step is the common hit: forward and backward of one step share it)."""
    key = (tuple(int(c) for c in counts), bool(use_bg), int(world), None if owners is None else tuple(int(o) for o in owners),
           int(hp), int(wp), int(chunk or shard_chunk_points(sum(int(c) for c in counts), world)))
    return _cached_plan(_plan_cache, key, lambda: ShardPlan(counts, use_bg, world, owners, hp, wp, key[-1]))


# ------------------------------------------------------------------------------------------------------ communicators
class _DeviceBytes:
    """A raw device allocation seen as a torch uint8 tensor (no copy) through __cuda_array_interface__."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def _as_tensor(ptr, nbytes, device):
    return torch.as_tensor(_DeviceBytes(ptr, nbytes), device=device)


class IpcComm:
    """One process per GPU (torchrun): the workspaces are cudaMalloc'ed, their CUDA IPC handles are exchanged over the
    process group once (all_gather_object), and every rank maps its peers' workspaces (dgvcc_peer_open).  After that
    the data path never touches the process group."""

    def __init__(self, group=None, device=None, nbytes=512 << 20):
        import torch.distributed as dist
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.nbytes = int(nbytes)
        lib = _native.lib()
        with torch.cuda.device(self.device):
            own = ctypes.c_void_p()
            _native.check(lib.dgvcc_peer_alloc(self.nbytes, ctypes.byref(own)), "dgvcc_peer_alloc")
            handle = (ctypes.c_ubyte * 64)()
            _native.check(lib.dgvcc_peer_export(own, handle), "dgvcc_peer_export")
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(handle), group=group)
            self.ptrs = []
            for r, h in enumerate(handles):
                if r == self.rank:
                    self.ptrs.append(own.value)
                    continue
                p = ctypes.c_void_p()
                buf = (ctypes.c_ubyte * 64).from_buffer_copy(h)
                _native.check(lib.dgvcc_peer_open(buf, ctypes.byref(p)), f"dgvcc_peer_open(rank {r})")
                self.ptrs.append(p.value)
            dist.barrier(group=group)
        self._finish()

    def close(self):
        """Unmap the peers' workspaces and free this rank's own (collective in spirit: call it on every rank, after the
        last step has been synchronised)."""
        if getattr(self, "ptrs", None) is None or isinstance(self, LocalComm):
            return
        torch.cuda.synchronize(self.device)
        lib = _native.lib()
        self.workspace = self.peer_table = None
        with torch.cuda.device(self.device):
            for r, p in enumerate(self.ptrs):
                if r != self.rank:
                    lib.dgvcc_peer_close(ctypes.c_void_p(p))
            import torch.distributed as dist
            if dist.is_initialized():
                dist.barrier(group=self.group)   # nobody frees memory a peer still has mapped and may be writing to
            lib.dgvcc_peer_free(ctypes.c_void_p(self.ptrs[self.rank]))
        self.ptrs = None

    def _finish(self):
        with torch.cuda.device(self.device):
            _native.check(_native.lib().dgvcc_bl_shard_preload(), "dgvcc_bl_shard_preload")
        self.workspace = _as_tensor(self.ptrs[self.rank], self.nbytes, self.device)
        self.peer_table = torch.tensor(self.ptrs, dtype=torch.int64, device=self.device)
        self.epoch = 0
        self.fuse_waits = not isinstance(self, LocalComm)   # ranks that share one GPU need the one-warp wait kernels


class LocalComm(IpcComm):
    """``world`` ranks inside ONE process on one GPU (tests, single-GPU development): plain allocations, plain pointers."""

    def __init__(self, rank, world, buffers):
        self.group, self.rank, self.world = None, rank, world
        self.device, self.nbytes = buffers[0].device, buffers[0].numel()
        self.ptrs = [b.data_ptr() for b in buffers]
        self._buffers = buffers
        self._finish()

    @staticmethod
    def make(world, device, nbytes=256 << 20):
        buffers = [torch.zeros(nbytes, dtype=torch.uint8, device=device) for _ in range(world)]
        return [LocalComm(r, world, buffers) for r in range(world)]


# ------------------------------------------------------------------------------------------------------------ autograd
class _PeerFn(torch.autograd.Function):
    """One rank's forward / backward of either peer split; the native launches are the module's ``_forward`` /
    ``_backward`` (one ctypes call each)."""

    @staticmethod
    def forward(ctx, density_local, mod, plan, packed, st, inv_batch):
        comm = mod.comm
        dev, r = comm.device, comm.rank
        _native.require_cuda(st, f"{type(mod).__name__}.forward")
        n_own = len(plan.owned[r])
        dens = density_local.detach().reshape(n_own, plan.hp, plan.wp).to(torch.float32).contiguous() if n_own else None
        if plan.layout.total > comm.nbytes:
            raise RuntimeError(f"sharded workspace of {comm.nbytes} bytes is too small for this batch ({plan.layout.total} "
                               "bytes); create the communicator with a larger nbytes")
        comm.epoch += 1
        shard = plan.shards[r]
        shard.epoch, shard.fuse_waits = comm.epoch, int(comm.fuse_waits)
        tables = plan.tables_on(r, dev)
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        deferred = mod._forward(plan, packed, st, dens, inv_batch, shard, tables, loss, ctx.needs_input_grad[0])
        ctx.saved = (mod, plan, packed, tables, inv_batch, comm.epoch, density_local.shape, density_local.dtype, n_own, deferred)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_loss):
        mod, plan, packed, tables, inv_batch, epoch, shape, dtype, n_own, deferred = ctx.saved
        comm = mod.comm
        dev = comm.device
        if epoch != comm.epoch:
            raise RuntimeError(f"{type(mod).__name__}: backward of a step whose shared workspace was already re-used by a "
                               "later forward (one forward/backward pair at a time per communicator)")
        shard = plan.shards[comm.rank]
        shard.epoch, shard.fuse_waits = epoch, int(comm.fuse_waits)
        g = grad_loss.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        grad = torch.empty((max(n_own, 1), plan.hp, plan.wp), dtype=torch.float32, device=dev)
        mod._backward(plan, packed, inv_batch, g, shard, tables, grad, deferred)
        return (grad[:n_own].reshape(shape).to(dtype),) + (None,) * 5


class _PackedAll:
    """Points / targets of the whole batch on the device plus this rank's table (one pinned upload)."""

    def __init__(self, points, targets, plan, rank, device):
        meta = plan.meta_for(rank)
        o_pts, o_tgt, total = _bl._pack_into(None, meta, points, targets, plan.total_points)
        host = torch.empty((total,), dtype=torch.uint8, pin_memory=True)
        _bl._pack_into(host.numpy(), meta, points, targets, plan.total_points)
        buf = host.to(device, non_blocking=True)
        n = max(plan.total_points, 1)
        self.meta = buf[:meta.nbytes].view(torch.int32)
        self.pts = buf[o_pts:o_pts + 8 * n].view(torch.float32).view(-1, 2)
        self.targets = buf[o_tgt:o_tgt + 4 * n].view(torch.float32)


class _PeerBL(Module):
    """What both peer splits of ``BL`` share: the forward (plan, re-pack cache, ``_PeerFn``), the per-phase timing and
    the error check.  A split supplies ``_plan``, the launches ``_forward`` / ``_backward`` and the names of the phases
    its launches time (``FWD_PHASES`` / ``BWD_PHASES``: one event before each phase and one after the last)."""

    def __init__(self, sigma, c_size, stride, background_ratio, use_background, device, comm):
        super().__init__()
        self.post_prob = _bl.Post_Prob(sigma, c_size, stride, background_ratio, use_background, device)
        self.bay_loss = _bl.Bay_Loss(use_background, device)
        self.comm = comm
        self.exact_cull = True
        self._last = None   # (key, packed): a benchmark / test that feeds the same lists again skips the re-pack

    def forward(self, points, st_sizes, target_list, pre_density_local, owners=None):
        comm = self.comm
        dev = comm.device
        points = _bl._as_point_list(points)
        counts = [int(p.shape[0]) for p in points]
        hp, wp = int(pre_density_local.shape[-2]), int(pre_density_local.shape[-1])
        plan = self._plan(counts, owners, hp, wp)
        if pre_density_local.shape[0] != len(plan.owned[comm.rank]):
            raise ValueError(f"rank {comm.rank} owns {len(plan.owned[comm.rank])} images of this batch but was given "
                             f"{pre_density_local.shape[0]} density maps")
        key = (id(plan), tuple(id(p) for p in points), tuple(id(t) for t in target_list))
        if self._last is not None and self._last[0] == key:
            packed = self._last[1]
        else:
            packed = _PackedAll(points, target_list, plan, comm.rank, dev)
            self._last = (key, packed, points, target_list)   # the lists are kept alive so that the ids stay meaningful
        st = st_sizes.to(device=dev, dtype=torch.float32).contiguous()
        return _PeerFn.apply(pre_density_local, self, plan, packed, st, 1.0 / plan.batch)

    def _event_handles(self, which):
        """None, or ctypes array of cudaEvent_t for the per-phase timing (``profile = True``)."""
        if not getattr(self, "profile", False):
            return None
        n = len(self.FWD_PHASES if which == "fwd" else self.BWD_PHASES) + 1
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n)]
        for e in evs:
            e.record()  # materialises the handle
        self._events = getattr(self, "_events", {})
        self._events[which] = evs
        return (ctypes.c_void_p * n)(*[e.cuda_event for e in evs])

    def phase_ms(self):
        """{phase: ms} of the last profiled step (synchronises)."""
        torch.cuda.synchronize(self.comm.device)
        out = {}
        for which, names in (("fwd", self.FWD_PHASES), ("bwd", self.BWD_PHASES)):
            evs = self._events[which]
            for k, name in enumerate(names):
                out[f"{which}: {name}"] = evs[k].elapsed_time(evs[k + 1])
        return out

    def check(self):
        """Synchronise and raise if a wait of the exchange protocol timed out (a peer died or fell out of step)."""
        torch.cuda.synchronize(self.comm.device)
        off = plan_err_offset(self.comm.world)
        err = int(self.comm.workspace[off:off + 4].view(torch.int32).item())
        if err:
            ph, src = (err - 1) % 16, (err - 1) // 16
            raise RuntimeError(f"{type(self).__name__} rank {self.comm.rank}: no flag of phase {ph} from rank {src} within 2 s")


class ChunkShardedBL(_PeerBL):
    """``BL`` for one batch spread over ``comm.world`` GPUs by point chunks (module docstring)."""

    FWD_PHASES = ["issue DENS copy (side stream)", "grid build + minima", "z (+Z out)", "[wait Z, DENS] finish_z", "counts",
                  "reduce_counts (+CNT out)", "[wait CNT] select (+LOSS out)", "[wait LOSS] loss"]
    BWD_PHASES = ["grad (+GPART out)", "[wait GPART] reduce (+GRAD out)", "[wait GRAD] gather", "[wait LOSS] deferred loss"]

    def __init__(self, sigma, c_size, stride, background_ratio, use_background, device, comm):
        super().__init__(sigma, c_size, stride, background_ratio, use_background, device, comm)
        # The images' losses come from all ranks: waiting for them is a barrier over the whole group that the backward pass
        # does not need.  With defer_loss (and a backward pass to follow) the forward returns at once and the backward
        # launches close with that wait: the returned tensor holds the loss once ``backward()`` has been called --
        # the usual order of a training step (``loss.backward(); loss.item()``).  False: complete after forward.
        self.defer_loss = False

    def _plan(self, counts, owners, hp, wp):
        return plan_shards(counts, self.post_prob.use_bg, self.comm.world, owners, hp, wp)

    def _forward(self, plan, packed, st, dens, inv_batch, shard, tables, loss, backward_follows):
        """dgvcc_bl_shard_forward; returns ``loss`` when the backward pass is to complete it (defer_loss), else None."""
        comm, pp = self.comm, self.post_prob
        defer = bool(self.defer_loss and backward_follows)   # the backward pass carries the closing launches
        rc = _native.lib().dgvcc_bl_shard_forward(
            _native.ptr(packed.pts), _native.ptr(packed.targets), _native.ptr(packed.meta), _native.ptr(st), _native.ptr(dens),
            plan.batch, plan.hp, plan.wp, plan.total_rows, plan.total_chunks, plan.multi_chunk, float(pp.stride),
            float(pp.sigma), float(pp.bg_ratio), int(pp.use_bg), int(self.exact_cull), inv_batch, ctypes.byref(shard),
            _native.ptr(tables[0]), _native.ptr(tables[1]), _native.ptr(comm.peer_table), _native.ptr(comm.workspace),
            comm.nbytes, _native.ptr(loss), int(defer), _native.stream_ptr(comm.device), self._event_handles("fwd"))
        _native.check(rc, "dgvcc_bl_shard_forward")
        return loss if defer else None

    def _backward(self, plan, packed, inv_batch, g, shard, tables, grad, deferred):
        comm, pp = self.comm, self.post_prob
        rc = _native.lib().dgvcc_bl_shard_backward(
            _native.ptr(packed.pts), _native.ptr(packed.meta), plan.batch, plan.hp, plan.wp, plan.total_rows,
            plan.total_chunks, float(pp.stride), float(pp.sigma), int(pp.use_bg), int(self.exact_cull), inv_batch,
            _native.ptr(g), ctypes.byref(shard), _native.ptr(tables[0]), _native.ptr(tables[1]), _native.ptr(comm.peer_table),
            _native.ptr(comm.workspace), comm.nbytes, _native.ptr(grad), _native.ptr(deferred),
            _native.stream_ptr(comm.device), self._event_handles("bwd"))
        _native.check(rc, "dgvcc_bl_shard_backward")


def plan_err_offset(world):
    lay = _native.BLLayout()
    _native.check(_native.lib().dgvcc_bl_shard_workspace_layout(1, 1, 1, 1, 1, world, lay), "dgvcc_bl_shard_workspace_layout")
    return int(lay.err)
