"""ISW module step on fp16 / bf16 feature maps: the native half path against the cast-based route (x.float() into the
fp32 modules, y rounded to the input dtype, .float() into the loss -- what autocast training paid before the half path)
and against fp32 input, on the three config-5 layers.  One JSON line per (shape, variant) to stdout and to --out.

Timed: the module step forward + backward (InstanceWhitening + instance_whitening_loss) eagerly and replayed as a CUDA
graph, and get_covariance_matrix alone (forward).  CUDA events around each step, L2 overwritten before each timed step
(the maps fit in the 126 MB L2), the variants alternate inside every repetition.  Also reported: the bytes a step moves
by count of full-map passes (algorithmic, from shapes, not measured) and the memory held after the forward.

    python scripts/bench_isw_half.py [--reps 20] [--out profiles/r3_isw_half.jsonl]
"""
import argparse
import gc
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from dgvcc_b200.models.ISW import InstanceWhitening, get_covariance_matrix, instance_whitening_loss  # noqa: E402

SHAPES = [(8, 64, 160, 160), (8, 256, 80, 80), (8, 512, 40, 40)]
# HBM bytes per map element of one forward + backward step, counted as full-map passes of the kernels and casts:
#   fp32:      instnorm fwd 4+4, Gram 4, dX = S X 4+4, instnorm bwd (dy and y read twice) 8+8+4             = 40
#   half:      instnorm fwd 2+2, Gram 2, dX 2+2, instnorm bwd (dy and x read twice) 4+4+2                   = 20
#   restated:  x.float() 2+4, fp32 instnorm 8, .to(half) 4+2, .float() 2+4, Gram 4, dX 8, cast of dX 4+2,
#              cast of dy 2+4, fp32 instnorm bwd 20, cast of dx 4+2                                          = 76
BYTES_PER_ELEMENT = {"fp32": 40, "half": 20, "restated": 76}
VARIANTS = [("fp32", torch.float32), ("half", torch.float16), ("restated", torch.float16), ("half", torch.bfloat16),
            ("restated", torch.bfloat16)]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


class Case:
    def __init__(self, shape, kind, dtype, dev):
        b, c, h, w = shape
        self.kind, self.dtype = kind, dtype
        g = torch.Generator().manual_seed(0)
        self.x = torch.randn(shape, generator=g).to(dtype).to(dev).requires_grad_(True)
        self.mask = (torch.rand(c, c, generator=g) < 0.5).float().triu(1).to(dev)
        self.eye, self.nr = torch.eye(c, device=dev), self.mask.sum()
        self.iw = InstanceWhitening(c)

    def forward(self):
        if self.kind == "restated":
            y = self.iw(self.x.float())[1].to(self.dtype).float()
        else:
            y = self.iw(self.x)[1]
        return instance_whitening_loss(y, self.eye, self.mask, 0, self.nr)

    def step(self):
        self.x.grad = None
        loss = self.forward()
        loss.backward()
        return loss

    def covariance(self):
        with torch.no_grad():
            return get_covariance_matrix(self.x.float() if self.kind == "restated" else self.x)[0]

    def held_after_forward(self):
        self.x.grad = None
        gc.collect()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        loss = self.forward()
        torch.cuda.synchronize()
        held = torch.cuda.memory_allocated() - base
        del loss
        return held

    def capture(self):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                self.step()
        torch.cuda.current_stream().wait_stream(side)
        self.x.grad = None
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
    lines = []
    for shape in SHAPES:
        numel = shape[0] * shape[1] * shape[2] * shape[3]
        cases = [Case(shape, kind, dtype, dev) for kind, dtype in VARIANTS]
        held = [c.held_after_forward() for c in cases]
        for c in cases:
            for _ in range(3):
                c.step()
                c.covariance()
            c.capture()
        torch.cuda.synchronize()
        t = {i: {"eager": [], "graph": [], "cov": []} for i in range(len(cases))}
        for rep in range(args.reps):   # the variants alternate inside each repetition
            for i, c in enumerate(cases):
                t[i]["eager"].append(timed(c.step, flush))
                t[i]["graph"].append(timed(c.graph.replay, flush))
                t[i]["cov"].append(timed(c.covariance, flush))
        for i, c in enumerate(cases):
            med = {k: sorted(v)[len(v) // 2] for k, v in t[i].items()}
            bpe = BYTES_PER_ELEMENT[c.kind]
            line = {"workload": "isw_module_step", "shape": list(shape), "variant": c.kind,
                    "dtype": str(c.dtype).replace("torch.", ""), "eager_ms": round(med["eager"], 4),
                    "graph_ms": round(med["graph"], 4), "covariance_ms": round(med["cov"], 4),
                    "eager_ms_min": round(min(t[i]["eager"]), 4), "graph_ms_min": round(min(t[i]["graph"]), 4),
                    "algorithmic_bytes_per_element": bpe, "algorithmic_bytes": bpe * numel,
                    "graph_algorithmic_gbs": round(bpe * numel / (med["graph"] * 1e-3) / 1e9, 1),
                    "held_after_forward_bytes": held[i], "held_bytes_per_element": round(held[i] / numel, 3),
                    "reps": args.reps, "l2": "overwritten (256 MB) before each timed step", "timing": "median of CUDA events",
                    "gpu": gpu}
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
