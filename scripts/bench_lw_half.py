"""lw_loss and ortho_loss on fp16 / bf16 inputs: the native half route against the cast route (x.float() into the fp32
route, the gradient rounded back to the input dtype -- what autocast training paid before) and against fp32 input.
One JSON line per (workload, shape, variant) to stdout and to --out.

lw_loss runs on the three config-5 layers with and without a mask, ortho_loss on a few [C, P] banks.  Timed: the
forward + backward step eagerly and replayed as a CUDA graph, and the Gram alone (the fused standardise-on-load Gram of
the native lw route, dgvcc_isw_gram on the materialised map otherwise).  CUDA events around each step, L2 overwritten
before each timed step, the variants alternate inside every repetition, medians reported.  Also reported: the memory
held after the forward, and the bytes a step moves counted from the kernels' loops (algorithmic, not measured).

    python scripts/bench_lw_half.py [--reps 20] [--out profiles/r3_lw_half.jsonl]
"""
import argparse
import gc
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from dgvcc_b200 import _native  # noqa: E402
from dgvcc_b200.losses.lw import lw_loss  # noqa: E402
from dgvcc_b200.losses.ortho import ortho_loss  # noqa: E402

LW_SHAPES = [(8, 64, 160, 160), (8, 256, 80, 80), (8, 512, 40, 40)]
ORTHO_SHAPES = [(256, 6400), (512, 25600), (512, 102400)]
# HBM bytes per element of the map, one forward + backward step, counted as passes of the kernels' loops over the map
# (a plane read twice counts twice; mask reads counted where a loop reads the mask once per map element):
#   lw fp32:    standardise fwd: x 3x4, yhat 4 (+ masked map 4, mask 4); Gram y 4; dY = S Y: y 4 + dy 4;
#               standardise bwd: dy 2x4, yhat 2x4 (+ mask 2x4), dx 4                       = 48 (masked 64)
#   lw half:    statistics x 2x2; fused Gram x 2; fused dY x 2 + dy 4; bwd dy 2x4 (+ mask 2x4), x 2x2, dx 2
#                                                                                           = 26 (masked 34)
#   lw cast:    x.float() 2+4, the fp32 route, dx.to() 4+2                                 = 60 (masked 76)
#   ortho (per element of the stacked [x; y]):  fp32: cat 4+4, Gram 4, two dX 4+4 = 20; half: cat 2+2, Gram 2, dX 2+2
#               = 10; cast: .float() 2+4, cat 4+4, Gram 4, dX 4+4, .to() 4+2 = 32
BYTES_PER_ELEMENT = {("lw", False): {"fp32": 48, "native": 26, "cast": 60},
                     ("lw", True): {"fp32": 64, "native": 34, "cast": 76},
                     ("ortho", False): {"fp32": 20, "native": 10, "cast": 32}}
VARIANTS = [("fp32", torch.float32), ("native", torch.float16), ("cast", torch.float16), ("native", torch.bfloat16),
            ("cast", torch.bfloat16)]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


class Case:
    def __init__(self, workload, shape, masked, kind, dtype, dev):
        self.workload, self.kind, self.dtype = workload, kind, dtype
        g = torch.Generator().manual_seed(0)
        self.mask = None
        if workload == "lw":
            self.inputs = [torch.randn(shape, generator=g).to(dtype).to(dev).requires_grad_(True)]
            if masked:
                b, _, h, w = shape
                self.mask = torch.rand((b, 1, h, w), generator=g).to(dev)
        else:
            self.inputs = [torch.randn(shape, generator=g).to(dtype).to(dev).requires_grad_(True) for _ in range(2)]
        self._gram_setup(dev)

    def forward(self):
        xs = [x.float() for x in self.inputs] if self.kind == "cast" else self.inputs
        return lw_loss(xs[0], self.mask) if self.workload == "lw" else ortho_loss(*xs)

    def step(self):
        for x in self.inputs:
            x.grad = None
        loss = self.forward()
        loss.backward()
        return loss

    def _gram_setup(self, dev):
        """Buffers of the forward's Gram call alone."""
        lib, P = _native.lib(), _native.ptr
        x = self.inputs[0].detach()
        if self.workload == "lw":
            n, c, h, w = x.shape
            hw = h * w
            m = self.mask.reshape(n, hw).contiguous() if self.mask is not None else None
            self.keep = [m]
        else:
            z = torch.cat([t.detach() for t in self.inputs])
            n, c, hw = 1, z.shape[0], z.shape[1]
            self.keep = [z]
        nbytes = lib.dgvcc_isw_workspace_bytes(n, c, hw)
        ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        gram = torch.empty((n, c, c), device=dev)
        self.keep += [ws, gram]
        st = _native.stream_ptr(dev)
        code = {torch.float16: _native.DTYPE_F16, torch.bfloat16: _native.DTYPE_BF16}.get(self.dtype)
        if self.kind == "native" and self.workload == "lw":
            stats = torch.empty((3, n * c), device=dev)
            self.keep.append(stats)
            _native.check(lib.dgvcc_lw_standardize_stats_h(P(x), code, n, c, hw, 1e-5, P(stats[0]), P(stats[1]), P(stats[2]),
                                                           st), "stats")
            self.gram = lambda: _native.check(lib.dgvcc_lw_gram_h(P(x), code, P(stats[0]), P(stats[1]), P(m), n, c, hw,
                                                                  P(ws), nbytes, P(gram), st), "dgvcc_lw_gram_h")
        elif self.kind == "native":
            self.gram = lambda: _native.check(lib.dgvcc_isw_gram_h(P(z), code, 1, c, hw, P(ws), nbytes, P(gram), st),
                                              "dgvcc_isw_gram_h")
        else:   # fp32 and cast routes: the fp32 Gram on the materialised fp32 operand
            if self.workload == "lw":
                y = torch.empty((n, c, hw), device=dev)
                ym = torch.empty_like(y) if m is not None else None
                inv = torch.empty((n * c,), device=dev)
                _native.check(lib.dgvcc_lw_standardize_forward(P(x.float().contiguous()), P(m), n, c, hw, 1e-5, P(y), P(ym),
                                                               P(inv), st), "fwd")
                y = ym if m is not None else y
            else:
                y = z.float()
            self.keep.append(y)
            self.gram = lambda: _native.check(lib.dgvcc_isw_gram(P(y), n, c, hw, 1, P(ws), nbytes, P(gram), st),
                                              "dgvcc_isw_gram")

    def held_after_forward(self):
        for x in self.inputs:
            x.grad = None
        gc.collect()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        loss = self.forward()
        torch.cuda.synchronize()
        held = torch.cuda.memory_allocated() - base
        route = getattr(loss.grad_fn, "half", None) if self.kind == "native" else None
        del loss
        return held, route

    def capture(self):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self.step()
        torch.cuda.current_stream().wait_stream(side)
        for x in self.inputs:
            x.grad = None
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = self.forward()
            self.loss.backward()


def timed(fn, flush):
    flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    gpu = gpu_info()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    groups = [("lw", s, m) for s in LW_SHAPES for m in (False, True)] + [("ortho", s, False) for s in ORTHO_SHAPES]
    lines = []
    for workload, shape, masked in groups:
        numel = 1
        for d in shape:
            numel *= d
        if workload == "ortho":
            numel *= 2
        cases = [Case(workload, shape, masked, kind, dtype, dev) for kind, dtype in VARIANTS]
        held = [c.held_after_forward() for c in cases]
        for c in cases:
            for _ in range(3):
                c.step()
                c.gram()
            c.capture()
        torch.cuda.synchronize()
        t = {i: {"eager": [], "graph": [], "gram": []} for i in range(len(cases))}
        for rep in range(args.reps):   # the variants alternate inside each repetition
            for i, c in enumerate(cases):
                t[i]["eager"].append(timed(c.step, flush))
                t[i]["graph"].append(timed(c.graph.replay, flush))
                t[i]["gram"].append(timed(c.gram, flush))
        for i, c in enumerate(cases):
            med = {k: sorted(v)[len(v) // 2] for k, v in t[i].items()}
            bpe = BYTES_PER_ELEMENT[(workload, masked)][c.kind]
            line = {"workload": f"{workload}_loss_step", "shape": list(shape), "masked": masked, "variant": c.kind,
                    "dtype": str(c.dtype).replace("torch.", ""), "native_route_taken": held[i][1] is not None,
                    "eager_ms": round(med["eager"], 4), "graph_ms": round(med["graph"], 4), "gram_ms": round(med["gram"], 4),
                    "eager_ms_min": round(min(t[i]["eager"]), 4), "graph_ms_min": round(min(t[i]["graph"]), 4),
                    "counted_bytes_per_element": bpe, "counted_bytes": bpe * numel,
                    "graph_counted_gbs": round(bpe * numel / (med["graph"] * 1e-3) / 1e9, 1),
                    "held_after_forward_bytes": held[i][0], "held_bytes_per_element": round(held[i][0] / numel, 3),
                    "reps": args.reps, "l2": "overwritten (256 MB) before each timed step",
                    "timing": "median of CUDA events", "gpu": gpu}
            lines.append(line)
            print(json.dumps(line), flush=True)
        del cases
        gc.collect()
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
