"""bench.py -- Bayesian-loss fwd+bwd images/s on the QNRF-shaped workload (BASELINE.json).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        # the UNMODIFIED reference losses/bl.py on the host cores (oracle/_ref)
    python bench.py ... --dump-outputs DIR      # also save loss.npy / density_grad.npy of the last timed step

One "step" = one pass of the hot path (BL forward + backward) over one batch of 16 synthetic
QNRF-shaped images per GPU (2048x1536 px, stride-8 grid 192x256, 500..12000 heads, CSR-packed).
Images are sharded across ranks (weak scaling: 16 images per GPU); the only collective is the
all-reduce of the scalar loss.  Prints ONE JSON line on rank 0.

  value     images/s, inputs already resident in HBM, through the drop-in ``BL`` module (dense sweep)
  e2e       images/s with HOST inputs: packed H2D copies of points/targets/density/st_sizes and
            D2H of the loss and the density gradient inside the timed region
  roofline  the fused path's MUFU.EX2 work (3 exponentials per point-pixel pair, dense) against the
            chip's MUFU.EX2 rate measured live by dgvcc_probe_ex2 (MEASURED_PEAKS.json has no
            SFU figure); per-kernel shares from CUDA events recorded on the launch stream
  cpu_baseline  the unmodified reference on the host cores: ONE full step over the same 16 images
  gpu_eager     the unmodified reference module with device='cuda' on the same B200 (PyTorch eager)
  strong    (N > 1) the SAME 16-image batch spread over the N GPUs: by image (snake partition) and by
            point chunk (sub-image sharding over NVLink peer memory), speed-up over one GPU
  aux       the two other north-star kernels: Gaussian splat (HBM roofline) and ISW Gram (tensor roofline)
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CONFIG = 3
STRIDE, SIGMA, BG_RATIO, USE_BG = 8, 8.0, 1.0, True
IMAGES_PER_GPU = 16


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=240.0,
                    help="wall budget of the --impl reference arm (it stops early, reporting the steps it ran)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true", help="skip the splat / Gram lines")
    ap.add_argument("--no-eager", action="store_true", help="skip the PyTorch-eager-on-GPU reference leg")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling legs at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and density gradient of the last timed step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def dump_outputs(out_dir, arrays):
    """Save float32 / float64 arrays as ``out_dir/<name>.npy``; the inputs are seeded, so two builds can be compared."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def workload(rank):
    from dgvcc_b200 import synthetic
    counts = synthetic.config_counts(CONFIG, IMAGES_PER_GPU)
    w, h = synthetic.CONFIG_SHAPES[CONFIG]
    pts, tgt, dens, st = synthetic.bl_batch(CONFIG, counts, w, h, STRIDE, first_image=rank * IMAGES_PER_GPU)
    return {
        "counts": counts, "width": w, "height": h, "hp": h // STRIDE, "wp": w // STRIDE,
        "points": [torch.from_numpy(p) for p in pts], "targets": [torch.from_numpy(t) for t in tgt],
        "density": torch.from_numpy(dens), "st_sizes": torch.from_numpy(st),
    }


def workload_name(wl):
    return (f"BASELINE config 3: {IMAGES_PER_GPU} QNRF-shaped images per GPU, {wl['width']}x{wl['height']} px, "
            f"stride-{STRIDE} grid {wl['hp']}x{wl['wp']}, {min(wl['counts'])}..{max(wl['counts'])} heads "
            f"({sum(wl['counts'])} per batch), sigma={SIGMA}, background on")


# ----------------------------------------------------------------------------- CPU reference arm
def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    torch.set_num_threads(max(1, n))


class ReferenceBL:
    """The reference's own Bayesian loss on ``device``: the UNMODIFIED losses/bl.py from oracle/_ref (byte copy made by
    oracle/make_ref.sh; /root/reference itself does not exist on the GPU box), else the oracle port.

    losses/bl.py is square-only (one ``cood`` vector for x and y, bl.py:14-16) and concatenates the batch before it
    splits it (bl.py:21-35: [sum N, M] temporaries, ~40 GB for this batch), so the module is called the way SURVEY 8c
    prescribes: c_size = max(H, W) = 2048, the 192x256 density zero-padded to the 256x256 grid (zero density adds
    exactly nothing to any count), one image per call, losses summed / B.  That is 33 % more pixels than the B200 arm
    evaluates -- the cost of running the reference unmodified on a non-square image."""

    def __init__(self, wl, device):
        self.wl, self.device = wl, torch.device(device)
        self.kind, self.mod = "port", None
        try:
            from oracle import ref_loader
            if ref_loader.available("bl"):
                c = max(wl["width"], wl["height"])
                self.mod = ref_loader.load("bl").BL(SIGMA, c, STRIDE, BG_RATIO, USE_BG, self.device)
                self.kind, self.side = "reference", c // STRIDE
        except Exception as exc:  # fall back to the port, say why
            self.note = f"unmodified reference not usable ({type(exc).__name__}: {exc}); oracle port timed instead"
        dev = self.device
        self.pts = [p.to(dev) for p in wl["points"]]
        self.tgt = [t.to(dev) for t in wl["targets"]]
        self.st = wl["st_sizes"].to(dev)
        self.dens = wl["density"].to(dev)

    def describe(self):
        if self.kind == "reference":
            return ("unmodified losses/bl.py (oracle/_ref), image by image, c_size=2048: the 192x256 density zero-padded to "
                    "the square 256x256 grid the reference needs")
        return "oracle port of losses/bl.py (oracle/bl_oracle.py), image by image on the 192x256 grid"

    def step(self):
        """One forward + backward over the whole batch; returns (seconds, loss)."""
        wl, b = self.wl, len(self.wl["counts"])
        sync = (lambda: torch.cuda.synchronize(self.device)) if self.device.type == "cuda" else (lambda: None)
        sync()
        t0 = time.perf_counter()
        total = 0.0
        if self.kind == "reference":
            for i in range(b):
                d = torch.zeros((1, 1, self.side, self.side), dtype=torch.float32, device=self.device)
                d[0, 0, :wl["hp"], :wl["wp"]] = self.dens[i, 0]
                d.requires_grad_(True)
                loss = self.mod([self.pts[i]], self.st[i:i + 1], [self.tgt[i]], d) / b
                loss.backward()
                total += float(loss.detach())
                del d, loss
        else:
            from oracle import bl_oracle
            for i in range(b):
                l, _, _ = bl_oracle.bl_forward_backward([self.pts[i]], self.st[i:i + 1], [self.tgt[i]], self.dens[i:i + 1],
                                                        STRIDE, SIGMA, BG_RATIO, USE_BG)
                total += float(l) / b
        sync()
        return time.perf_counter() - t0, total


def cpu_baseline(wl):
    """ONE full step of the reference on the host cores (about 5-10 s on the box's 16 cores)."""
    use_all_host_threads()
    ref = ReferenceBL(wl, "cpu")
    dt, loss = ref.step()
    return {
        "value": len(wl["counts"]) / dt, "unit": "images/s", "cores": torch.get_num_threads(), "kind": ref.kind,
        "sample": f"{ref.describe()}; torch CPU, {torch.get_num_threads()} threads; ONE full forward+backward over the same "
                  f"16 images ({sum(wl['counts'])} heads) in {dt:.2f} s, nothing extrapolated",
        "loss": loss,
    }


def gpu_eager(wl, dev, reps=2):
    """SURVEY section 2's bar: the unmodified reference module as PyTorch eager ops on the SAME B200 (device='cuda')."""
    ref = ReferenceBL(wl, dev)
    ref.step()  # allocator warm-up
    times = [ref.step() for _ in range(reps)]
    dt = min(t for t, _ in times)
    out = {"value": len(wl["counts"]) / dt, "unit": "images/s", "kind": ref.kind, "ms_per_step": dt * 1e3,
           "loss": times[-1][1],
           "note": f"{ref.describe()}; torch CUDA eager on this GPU, best of {reps} full steps (wall clock around a synchronize)"}
    del ref
    torch.cuda.empty_cache()
    return out


def run_reference(args, emit=print):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    use_all_host_threads()
    wl = workload(0)
    ref = ReferenceBL(wl, "cpu")
    t_start = time.perf_counter()
    for _ in range(min(args.warmup, 1)):
        ref.step()
    times = []
    for _ in range(max(1, args.steps)):
        times.append(ref.step()[0])
        if time.perf_counter() - t_start > args.cpu_seconds:  # wall budget: report the steps actually run
            break
    per_batch = float(np.mean(times))
    value = len(wl["counts"]) / per_batch
    sample = (f"{ref.describe()}; torch CPU, {torch.get_num_threads()} threads; every step is the FULL 16-image batch "
              f"({sum(wl['counts'])} heads); {len(times)} of the {args.steps} requested steps fitted the {args.cpu_seconds:.0f} s budget")
    emit(json.dumps({
        "impl": "reference", "metric": "Bayesian-loss fwd+bwd images/s (QNRF shape)", "value": value,
        "unit": "images/s", "n_gpus": args.gpus, "steps": len(times), "steps_requested": args.steps,
        "warmup": min(args.warmup, 1), "ms_per_step": per_batch * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": workload_name(wl)},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": torch.get_num_threads(), "kind": ref.kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def profiled_dram_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the three sweep kernels (per launch each, summed: they are
    the path's exponential-carrying kernels), from the newest committed `ncu --set full` capture of this workload
    (profiles/r*_bl_ncu_raw.csv); None when no capture is in the tree."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r*_bl_ncu_raw.csv")))
    if not files:
        return None, "no ncu capture under profiles/"
    rows = list(csv.reader(open(files[-1])))
    hdr, units, data = rows[0], rows[1], rows[2:]
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total, per = 0.0, {}
    for r in data:
        name = r[hdr.index("Kernel Name")].split("(")[0].replace("void ", "").split("<")[0]
        if name not in ("bl_z_kernel", "bl_counts_kernel", "bl_grad_kernel"):
            continue
        b = 0.0
        for col in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            k = hdr.index(col)
            b += float(r[k].replace(",", "")) * scale.get(units[k], 1.0)
        per[name] = b
        total += b
    note = (f"{os.path.basename(files[-1])}: " + ", ".join(f"{k} {v / 1e6:.1f} MB" for k, v in per.items()) +
            "; against ~6 MB of algorithmic inputs/outputs per step the sweeps are nowhere near HBM-bound (MUFU-bound)")
    return total, note


# ----------------------------------------------------------------------------------- GPU arm
class ClockSampler:
    """SM clock and throttle reasons DURING the run, from two sources at once: `nvidia-smi -lms 100` in a subprocess (the
    profiling recipe's line) and an NVML thread in this process sampling every 20 ms (the timed region of a 1-GPU run is
    ~40 ms -- VERDICT r1: "only 4 clock samples fall under load").  Either source alone is enough; every failure of the
    NVML path is swallowed (the subprocess remains)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml_sm, self.nvml_bits, self.nvml_max, self.nvml_stop = [], 0, None, threading.Event()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None
        threading.Thread(target=self._nvml_loop, daemon=True).start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def _nvml_loop(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            try:  # the CUDA ordinal and the NVML index differ under CUDA_VISIBLE_DEVICES: go by UUID when torch has it
                handle = pynvml.nvmlDeviceGetHandleByUUID(f"GPU-{torch.cuda.get_device_properties(self.index).uuid}")
            except Exception:
                handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            self.nvml_max = float(pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM))
            while not self.nvml_stop.is_set():
                self.nvml_sm.append(float(pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)))
                self.nvml_bits |= int(reasons(handle))
                self.nvml_stop.wait(0.02)
        except Exception:
            pass

    def stop(self):
        self.nvml_stop.set()
        sm, reasons, mx = list(self.nvml_sm), set(), self.nvml_max
        for bit, name in self.NVML_REASONS.items():
            if self.nvml_bits & bit:
                reasons.add(name)
        n_nvml = len(sm)
        if self.proc is None and not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
            except ValueError:
                continue
            for name, val in zip(names, r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "samples_nvml_20ms": n_nvml, "samples_nvidia_smi_100ms": len(sm) - n_nvml}


def probe_peak(fn_name, dev, iters=20000):
    from dgvcc_b200 import _native
    fn = getattr(_native.lib(), fn_name)
    sink = torch.zeros(4, device=dev)
    ops = ctypes.c_int64(0)
    best = 0.0
    for rep in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _native.check(fn(_native.ptr(sink), iters, ctypes.byref(ops), _native.stream_ptr(dev)), fn_name)
        e1.record()
        torch.cuda.synchronize(dev)
        if rep:
            best = max(best, ops.value / (e0.elapsed_time(e1) * 1e-3))
    return best


def kernel_breakdown(wl, dev, reps=5):
    """Per-kernel device time of the fused path: CUDA events recorded on the launch stream between the
    launches of dgvcc_bl_forward_profiled / dgvcc_bl_backward (inputs resident, no host glue)."""
    from dgvcc_b200 import _native
    from dgvcc_b200.losses import bl as blmod
    lib = _native.lib()
    packed = blmod._Packed([p.to(dev) for p in wl["points"]], USE_BG, dev)
    targets = blmod._pack_targets([t.to(dev) for t in wl["targets"]], packed, dev)
    dens = wl["density"].to(dev).reshape(len(wl["counts"]), wl["hp"], wl["wp"]).contiguous()
    st = wl["st_sizes"].to(dev)
    b, hp, wp = dens.shape
    lay = blmod._layout(packed.total_rows, packed.total_chunks, b, hp, wp)
    ws = blmod._workspace(lay, dev)
    loss = torch.empty(1, device=dev)
    grad = torch.empty_like(dens)
    gl = torch.ones(1, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    names = ["bl_grid_build+bl_gridmin", "bl_z(+finish)", "bl_counts", "bl_reduce_counts+bl_select", "bl_grad(+finish)"]
    acc = np.zeros(len(names))
    for rep in range(reps + 1):
        flush.zero_()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        for e in ev:
            e.record()  # materialise the handles
        handles = (ctypes.c_void_p * 5)(*[e.cuda_event for e in ev[:5]])
        _native.check(lib.dgvcc_bl_forward_profiled(
            _native.ptr(packed.pts), _native.ptr(targets), _native.ptr(packed.meta), _native.ptr(st),
            _native.ptr(dens), b, hp, wp, packed.total_rows, packed.total_chunks, packed.multi_chunk, float(STRIDE),
            SIGMA, BG_RATIO, int(USE_BG), 0, 1.0 / b, _native.ptr(ws), lay.total, _native.ptr(loss),
            _native.stream_ptr(dev), handles), "dgvcc_bl_forward_profiled")
        _native.check(lib.dgvcc_bl_backward(
            _native.ptr(packed.pts), _native.ptr(packed.meta), b, hp, wp, packed.total_rows, packed.total_chunks,
            packed.multi_chunk, float(STRIDE), SIGMA, int(USE_BG), 0, 1.0 / b, _native.ptr(gl), _native.ptr(ws),
            lay.total, _native.ptr(grad), _native.stream_ptr(dev)), "dgvcc_bl_backward")
        ev[5].record()
        torch.cuda.synchronize(dev)
        if rep:
            acc += np.array([ev[i].elapsed_time(ev[i + 1]) for i in range(5)])
    ms = acc / reps
    wsel = ws[lay.wsel:lay.wsel + 4 * packed.total_rows].view(torch.float32)
    kept_rows = int((wsel != 0).sum())
    return dict(zip(names, ms.tolist())), kept_rows, packed


def aux_lines(dev, cpu=True):
    """The two other north-star kernels in the driver-run line (VERDICT r1 item 2): Gaussian splat against the HBM
    roofline (BASELINE config 4) and the ISW Gram against the tensor / HBM roofline (config 5), each with e2e and a
    CPU baseline.  Implemented in scripts/bench_aux.py (also runnable on its own)."""
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import bench_aux
    bench_aux.dev = dev
    out = {}
    out.update(bench_aux.dmap_lines(cpu))
    tf32 = bench_aux.probe_tf32_peak(dev)
    out.update(bench_aux.isw_lines(cpu, tf32))
    out["tf32_peak_tflops"] = tf32 / 1e12
    return out


def strong_scaling(args, dev, rank, world, t1_ms, flush, barrier):
    """Strong scaling of BASELINE config 3 as written: ONE batch of 16 images spread over the N GPUs.

    by_image: whole images assigned to ranks by ``snake_partition`` (cost N_i * M); bounded by the biggest image.
    Every rank times its own shard with per-step CUDA events; the step time of the job is the max over ranks."""
    import torch.distributed as dist
    from dgvcc_b200.losses.bl import BL
    from dgvcc_b200.sharding import ShardedLoss, snake_partition
    wl = workload(0)  # the SAME 16 images on every rank
    b, m = len(wl["counts"]), wl["hp"] * wl["wp"]
    out = {"batch": b, "heads": sum(wl["counts"]), "t1_ms": t1_ms,
           "note": ("the same 16-image batch (the one rank 0 holds in the weak run) spread over the N GPUs; t1_ms = rank 0's "
                    "device time per step for the whole batch on ONE GPU, measured in this run; speedup = t1_ms / max over "
                    "ranks of the per-step device time")}
    t1 = torch.tensor([t1_ms], device=dev, dtype=torch.float64)
    dist.broadcast(t1, 0)
    t1_ms = out["t1_ms"] = float(t1[0])

    # ---- by image
    shards = snake_partition([n * m for n in wl["counts"]], world)
    mine = shards[rank]
    mod = BL(SIGMA, max(wl["width"], wl["height"]), STRIDE, BG_RATIO, USE_BG, dev)
    mod.exact_cull = False
    fn = ShardedLoss(mod, b)
    pts = [wl["points"][i].to(dev) for i in mine]
    tgt = [wl["targets"][i].to(dev) for i in mine]
    st = wl["st_sizes"][mine].to(dev)
    dens = wl["density"][mine].to(dev).requires_grad_(True)

    def step():
        dens.grad = None
        loss = fn(pts, st, tgt, dens)
        loss.backward()
        return loss

    def timed(step_fn):
        for _ in range(3):
            step_fn()
            flush.zero_()
        barrier()
        evs = []
        for _ in range(args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step_fn()
            e1.record()
            evs.append((e0, e1))
            flush.zero_()
        barrier()
        ms = sum(a.elapsed_time(c) for a, c in evs) / args.steps
        allms = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(allms, torch.tensor([ms], device=dev, dtype=torch.float64))
        return [float(x[0]) for x in allms]

    per_rank = timed(step)
    heads = [sum(wl["counts"][i] for i in s) for s in shards]
    out["by_image"] = {
        "partition": "snake_partition by N_i * M (whole images)", "heads_per_rank": heads,
        "ms_per_rank": per_rank, "ms_per_step": max(per_rank), "imbalance_max_over_mean": max(per_rank) / (sum(per_rank) / world),
        "images_per_s": b / (max(per_rank) * 1e-3), "speedup": t1_ms / max(per_rank),
        "bound_by_largest_shard": sum(wl["counts"]) / max(heads),
        "collective": "one all_reduce(sum) of the scalar loss per step (NCCL)"}
    del pts, tgt, dens

    # ---- by point chunk: every rank sweeps 1/N of the packed point sequence, partials travel over NVLink peer memory
    from dgvcc_b200.losses.bl_sharded import ChunkShardedBL, IpcComm, plan_shards
    comm = IpcComm(device=dev)
    cmod = ChunkShardedBL(SIGMA, max(wl["width"], wl["height"]), STRIDE, BG_RATIO, USE_BG, dev, comm)
    cmod.exact_cull = False
    cmod.defer_loss = True   # a training step calls loss.backward() before it reads the value
    plan = plan_shards(wl["counts"], USE_BG, world, None, wl["hp"], wl["wp"])
    local_d = wl["density"][plan.owned[rank]].to(dev).requires_grad_(True)
    st_all = wl["st_sizes"].to(dev)

    def chunk_step():
        local_d.grad = None
        loss = cmod(wl["points"], st_all, wl["targets"], local_d)
        loss.backward()
        return loss

    per_rank = timed(chunk_step)
    cmod.check()
    # parity inside the bench run: the sharded loss against this rank's own one-GPU evaluation of the same batch
    ref_mod = BL(SIGMA, max(wl["width"], wl["height"]), STRIDE, BG_RATIO, USE_BG, dev)
    ref_mod.exact_cull = False
    d_all = wl["density"].to(dev).requires_grad_(True)
    ref_loss = ref_mod([p.to(dev) for p in wl["points"]], st_all, [t.to(dev) for t in wl["targets"]], d_all)
    ref_loss.backward()
    got = chunk_step()
    rel_loss = abs(float(got) - float(ref_loss)) / abs(float(ref_loss))
    gref = d_all.grad[plan.owned[rank]].reshape(local_d.grad.shape)
    rel_grad = float((local_d.grad - gref).abs().max() / gref.abs().max()) if len(plan.owned[rank]) else 0.0
    worst = torch.tensor([rel_loss, rel_grad], device=dev, dtype=torch.float64)
    dist.all_reduce(worst, op=dist.ReduceOp.MAX)
    m4 = 4 * m
    sent = sum(int(v[2]) & 0xffffffff for r in range(world) for v in plan.slices[r][:plan.shards[r].push_first[7]])
    heads = [int(plan.c_cnt[plan.chunk_lo[r]:plan.chunk_hi[r]].sum()) for r in range(world)]
    out["by_chunk"] = {
        "partition": f"packed point sequence cut into {world} equal spans, chunks of <= 1024 points ({plan.total_chunks} chunks)",
        "heads_per_rank": heads, "ranks_per_image": [len(g) for g in plan.groups],
        "ms_per_rank": per_rank, "ms_per_step": max(per_rank), "imbalance_max_over_mean": max(per_rank) / (sum(per_rank) / world),
        "images_per_s": b / (max(per_rank) * 1e-3), "speedup": t1_ms / max(per_rank),
        "collective": ("none: per-chunk minima / denominator shares / gradient sums, row counts, density and finished "
                       "gradients are stored straight into the peers' workspaces over NVLink (CUDA IPC peer memory) with one "
                       "arrival flag per (phase, source); 7 exchange phases per step"),
        "bytes_pushed_per_step_all_ranks": sent,
        "parity_vs_one_gpu": {"loss_rel": float(worst[0]), "grad_rel_to_max": float(worst[1]),
                              "note": "against the ordinary BL module on one GPU (other chunk boundaries, so other rounding of the "
                                      "chunk-partial sums); bit-identity with the same chunk table is tested in "
                                      "tests/test_bl_sharded_gpu.py and scripts/shard_bl_multi_gpu.py"}}
    # ---- by row band: every rank sweeps ALL points over 1/N of the grid rows; one exchange (the count shares)
    try:
        from dgvcc_b200.losses.bl_banded import BandShardedBL, plan_bands
        bmod = BandShardedBL(SIGMA, max(wl["width"], wl["height"]), STRIDE, BG_RATIO, USE_BG, dev, comm)
        bmod.exact_cull = False
        bplan = plan_bands(wl["counts"], USE_BG, world, None, wl["hp"], wl["wp"])
        band_d = wl["density"][bplan.owned[rank]].to(dev).requires_grad_(True)

        def band_step():
            band_d.grad = None
            loss = bmod(wl["points"], st_all, wl["targets"], band_d)
            loss.backward()
            return loss

        per_rank = timed(band_step)
        bmod.check()
        got = band_step()
        rel_loss = abs(float(got) - float(ref_loss)) / abs(float(ref_loss))
        gref = d_all.grad[bplan.owned[rank]].reshape(band_d.grad.shape)
        rel_grad = float((band_d.grad - gref).abs().max() / gref.abs().max()) if len(bplan.owned[rank]) else 0.0
        everyone = [torch.zeros(1, device=dev) for _ in range(world)]
        dist.all_gather(everyone, got.detach().reshape(1))
        worst = torch.tensor([rel_loss, rel_grad], device=dev, dtype=torch.float64)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        bmod.profile = True
        acc = {}
        for _ in range(5):
            band_step()
            for k, v in bmod.phase_ms().items():
                acc[k] = acc.get(k, 0.0) + v / 5
            flush.zero_()
        bmod.profile = False
        phases = [None] * world
        dist.all_gather_object(phases, acc)
        sent = sum(int(v[2]) & 0xffffffff for r in range(world) for v in bplan.slices[r][:bplan.shards[r].push_first[7]]
                   if (int(v[2]) >> 32) != r)
        tile_r, tile_c = bplan.layout.rows_per_thread, bplan.layout.cols_per_thread
        col_blocks = -(-wl["wp"] // (32 * tile_c))
        part_rows = [-(-(-(-int(h - l) // tile_r) * col_blocks) // 4) for l, h in zip(bplan.band_lo, bplan.band_hi)]
        sent += sum(part_rows) * (world - 1) * 4 * bplan.total_rows                           # CNT: every partial row to every peer
        sent += sum(4 * wl["wp"] * (wl["hp"] - int(bplan.band_hi[o] - bplan.band_lo[o])) for o in bplan.owners)   # GRAD rows
        out["by_band"] = {
            "partition": (f"grid rows cut into {world} bands of whole pixel-tile rows "
                          f"({[int(h - l) for l, h in zip(bplan.band_lo, bplan.band_hi)]} rows); every rank sweeps all "
                          f"{sum(wl['counts'])} heads ({bplan.total_chunks} chunks of <= {bplan.chunk} points) over its band"),
            "pixel_tile_rows_cols": [bplan.layout.rows_per_thread, bplan.layout.cols_per_thread],
            "ms_per_rank": per_rank, "ms_per_step": max(per_rank), "imbalance_max_over_mean": max(per_rank) / (sum(per_rank) / world),
            "images_per_s": b / (max(per_rank) * 1e-3), "speedup": t1_ms / max(per_rank),
            "collective": ("none (no NCCL on the data path): density rows owner -> band rank on a side stream; the per-CTA partial "
                           "counts of a band stored on every rank by bl_counts itself over NVLink peer memory (the ONE "
                           "data-dependent exchange; added in pixel-tile order, so every rank gets the same loss bits as one "
                           "GPU); gradient rows stored at the image's owner by bl_grad itself; one arrival flag per (phase, source)"),
            "bytes_pushed_per_step_all_ranks": sent,
            "phase_ms_max_over_ranks": {k: round(max(ph[k] for ph in phases), 4) for k in phases[0]},
            "same_loss_bits_on_every_rank": all(torch.equal(v, everyone[0]) for v in everyone),
            "parity_vs_one_gpu": {"loss_rel": float(worst[0]), "grad_rel_to_max": float(worst[1]),
                                  "note": "against the ordinary BL module on one GPU (1024-point chunks there); with the same "
                                          "chunk table the gradient is bit-identical (tests/test_bl_sharded_gpu.py, "
                                          "scripts/shard_bl_multi_gpu.py --mode band)"}}
    except Exception as exc:  # keep the other legs
        out["by_band"] = {"error": f"{type(exc).__name__}: {exc}"}
    return out


def run_gpu(args, emit=print):
    import torch.distributed as dist
    from dgvcc_b200.losses.bl import BL
    from dgvcc_b200.sharding import ShardedLoss

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = workload(rank)
    b = len(wl["counts"])
    m = wl["hp"] * wl["wp"]
    global_batch = b * world

    loss_mod = BL(SIGMA, max(wl["width"], wl["height"]), STRIDE, BG_RATIO, USE_BG, dev)
    loss_mod.exact_cull = False  # the graded numbers (value / e2e / roofline) are the DENSE sweep; the product default culls
    loss_fn = ShardedLoss(loss_mod, global_batch) if world > 1 else loss_mod

    # ---- resident inputs ("value")
    pts_d = [p.to(dev) for p in wl["points"]]
    tgt_d = [t.to(dev) for t in wl["targets"]]
    st_d = wl["st_sizes"].to(dev)
    dens_d = wl["density"].to(dev).requires_grad_(True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_resident():
        dens_d.grad = None
        loss = loss_fn(pts_d, st_d, tgt_d, dens_d)
        loss.backward()
        return loss

    # ---- host inputs ("e2e"): pinned host buffers in, loss + gradient out
    pts_h = [p.pin_memory() for p in wl["points"]]
    tgt_h = [t.pin_memory() for t in wl["targets"]]
    st_h = wl["st_sizes"].pin_memory()
    dens_h = wl["density"].pin_memory()
    grad_h = torch.empty_like(wl["density"]).pin_memory()
    h2d = sum(p.numel() * 4 for p in pts_h) + sum(t.numel() * 4 for t in tgt_h) + st_h.numel() * 4 + dens_h.numel() * 4
    d2h = grad_h.numel() * 4 + 4

    def step_host():
        d = dens_h.to(dev, non_blocking=True).requires_grad_(True)
        loss = loss_fn(pts_h, st_h.to(dev, non_blocking=True), tgt_h, d)  # host lists: packed, one H2D each
        loss.backward()
        grad_h.copy_(d.grad, non_blocking=True)
        return float(loss.detach())  # D2H of the loss: synchronises the step

    # the same with the batch packed by the data pipeline (pack_batch in the collate function): one pinned buffer
    from dgvcc_b200.losses.bl import pack_batch
    packed_h = pack_batch(wl["points"], wl["targets"], use_background=USE_BG).pin_memory()

    def step_host_packed():
        d = dens_h.to(dev, non_blocking=True).requires_grad_(True)
        loss = loss_fn(packed_h, st_h.to(dev, non_blocking=True), None, d)
        loss.backward()
        grad_h.copy_(d.grad, non_blocking=True)
        return float(loss.detach())

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    sampler = ClockSampler(local)  # samples clocks / throttle reasons through warm-up, timed region and e2e
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
        flush.zero_()
    peak_ex2 = probe_peak("dgvcc_probe_ex2", dev)
    peak_ffma = probe_peak("dgvcc_probe_ffma", dev)
    barrier()
    t_wall0 = time.perf_counter()
    events = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = step_resident()
        e1.record()
        events.append((e0, e1))
        flush.zero_()  # L2 flush between timed steps, outside the per-step events
        # the loss's autograd node holds the step's workspace: kept alive, the next step would allocate a second one
        loss = loss.detach() if args.dump_outputs else None
    barrier()
    wall = time.perf_counter() - t_wall0
    total_ms = sum(a.elapsed_time(c) for a, c in events)
    if args.dump_outputs and rank == 0:   # the legs below overwrite the gradient
        dump_outputs(args.dump_outputs, {"loss": loss, "density_grad": dens_d.grad})

    # informational: the same steps with the opt-in exact-zero culling (bit-identical results, not graded)
    loss_mod.exact_cull = True
    for _ in range(3):
        step_resident()
    barrier()
    cull_events = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step_resident()
        e1.record()
        cull_events.append((e0, e1))
        flush.zero_()
    barrier()
    cull_ms = sum(a.elapsed_time(c) for a, c in cull_events)
    loss_mod.exact_cull = False

    # e2e (warm-up longer than the ring of pinned staging buffers, so that no cudaHostAlloc falls into the timed region)
    for _ in range(6):
        step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    barrier()
    e2e_s = time.perf_counter() - t0
    for _ in range(6):
        step_host_packed()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host_packed()
    barrier()
    e2e_packed_s = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None

    own_ms_per_step = total_ms / args.steps  # this rank's own 16 images on one GPU: the 1-GPU time of the strong legs
    if world > 1:
        t = torch.tensor([total_ms, e2e_s, cull_ms, e2e_packed_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s, cull_ms, e2e_packed_s = float(t[0]), float(t[1]), float(t[2]), float(t[3])

    strong = None
    if world > 1 and not args.no_strong:
        try:
            strong = strong_scaling(args, dev, rank, world, own_ms_per_step, flush, barrier)
        except Exception as exc:  # the strong legs must never take the headline line down with them
            strong = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        ms_per_step = total_ms / args.steps
        value = global_batch / (ms_per_step * 1e-3)
        kernels, kept_rows, packed = kernel_breakdown(wl, dev)
        pairs = sum(wl["counts"]) * m
        kept_frac = kept_rows / max(1, packed.total_rows)
        path_ms = sum(kernels.values())
        algorithmic = 3.0 * pairs                       # SURVEY 8d: 3 exponentials per pair, dense
        executed = (2.0 + kept_frac) * pairs            # backward skips the 10 % of rows the top-k trims
        achieved = executed / (path_ms * 1e-3)
        traffic, traffic_note = profiled_dram_traffic()
        out = {
            "metric": "Bayesian-loss fwd+bwd images/s (QNRF shape)", "value": value, "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(wl), "global_batch": global_batch, "parallelism": f"image-sharded x{world}",
                       "l2": "flushed between timed steps (256 MiB memset outside the per-step CUDA events)",
                       "timing": "per-step CUDA events on the launch stream, max over ranks",
                       "wall_s_incl_flush": wall},
            "clocks": clocks,
            "e2e": {"value": global_batch * args.steps / e2e_s, "unit": "images/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "gpu_launches": args.steps * 7,   # grid_build, gridmin, z, counts, reduce_counts, select | grad
            "e2e_packed_collate": {"value": global_batch * args.steps / e2e_packed_s, "unit": "images/s",
                                   "note": ("informational: same end-to-end step, but the ragged lists were packed once by "
                                            "pack_batch (what a collate_fn does in the DataLoader workers) instead of inside "
                                            "every timed step; H2D of the packed buffer / density and D2H of loss / gradient "
                                            "are still inside the timed region")},
            "exact_cull": {"value": global_batch / (cull_ms / args.steps * 1e-3), "unit": "images/s",
                           "ms_per_step": cull_ms / args.steps,
                           "note": ("informational, NOT the graded number: BL.exact_cull=True skips (point, pixel-tile) "
                                    "pairs whose exponentials are provably exact zeros; results bit-identical to the "
                                    "dense path that value / e2e / roofline measure")},
            "roofline": {
                "bound": "sfu", "achieved": achieved / 1e9, "peak": peak_ex2 / 1e9, "unit": "Gexp/s",
                "frac": achieved / peak_ex2, "traffic": traffic, "traffic_note": traffic_note,
                "note": ("fused BL path (bl_grid_build+bl_gridmin+bl_z+bl_counts+bl_reduce_counts+bl_select+bl_grad: 7 launches), MUFU.EX2-bound; achieved = executed "
                         "exponentials / sum of kernel times; peak = dgvcc_probe_ex2 measured in this run "
                         "(MEASURED_PEAKS.json carries no SFU peak)"),
                "algorithmic_exps_per_step": algorithmic, "executed_exps_per_step": executed,
                "path_ms": path_ms, "kernels_ms": kernels, "ffma_peak_tflops": 2 * peak_ffma / 1e12,
            },
        }
        if strong is not None:
            out["strong"] = strong
        if not args.no_eager:
            try:
                out["gpu_eager"] = gpu_eager(wl, dev)
            except Exception as exc:
                out["gpu_eager"] = {"error": f"{type(exc).__name__}: {exc}"}
        if not args.no_aux:
            try:
                out["aux"] = aux_lines(dev, cpu=not args.no_cpu_baseline)
            except Exception as exc:
                out["aux"] = {"error": f"{type(exc).__name__}: {exc}"}
        if not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(wl)
        emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


class StdoutToStderr:
    """Libraries (e.g. NCCL's version banner) write to fd 1; keep stdout for the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, line):
        sys.stdout.flush()
        os.write(self.saved, (line + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


if __name__ == "__main__":
    a = parse()
    with StdoutToStderr() as out:
        printer = lambda line: out.emit(line)  # noqa: E731
        if a.impl == "reference":
            run_reference(a, printer)
        else:
            run_gpu(a, printer)
