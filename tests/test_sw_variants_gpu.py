"""Switchable whitening (csrc/sw_kernels.cu) against the fp64 kernel-order restatement (oracle/switchwhiten_oracle.py:
``decomposed``) at every moments split plan, in every mode, and on off-centre planes.

The two moments passes stream each CTA's pixel chunk through a private ring of shared-memory slots (8 stages forward,
6 backward).  The host planner ``plan_split`` picks the chunk: as many CTAs per plane as one resident wave holds
(148 SMs x 2 / planes, the backward counting its z row blocks per plane: 2 at cp = 16, 1 at cp = 8 and 4), at most one
per 512 pixels, at least one.  PLAN_CASES names, for each shape, the arms it was built to reach -- which of the three
limits set the split count, how many ring iterations a CTA runs (stages - 1, stages, stages + 1, or three wraps and
more), what the last split holds (one pixel, under 128, a full chunk), and the plane-size edges (hw = 1, 2, < 128,
hw = 1 or 511 mod 512 for the partial affine CTA).  A restatement of the planner checks every case lands where its
tags say, and the library's workspace size (which grows with the split counts) checks the restatement.

Each GPU case runs the six C entry points one by one from a NaN-filled workspace and compares every stage with the
fp64 value of the same fp32 inputs: mean_in and cov_in (against two-pass statistics of x.double()), the batch mean and
covariance, the running buffers, a_fwd, y, the six outputs of backward_stats and grad_x.  Then the module runs the same
inputs and must reproduce those stages bit for bit.

OFFSET_CASES put a plane off centre, on a multi-split and on a one-split shape: pixel 0 of every channel of a group
10, 30 or 100 standard deviations away, a group constant except for pixel 0 (a rank-one covariance), and every channel
at a mean of 10 or 100 standard deviations.  The forward moments are centred on a sample mean of the plane; centred on
pixel 0, the first cases lose k^2 x 6e-8 of the covariance to cancellation.

Gates (those of test_sw_gpu.py against fp64): |got - ref| <= 2e-5 (|ref| + max|ref|), the max taken per (sample,
group) for mean_in, cov_in and a_fwd and over the whole tensor otherwise.  The reference's own fp32 evaluation
(oracle ``forward_backward``) is recorded as an (accuracy) margin beside the kernels'.
"""
import numpy as np
import pytest
import torch

from dgvcc_b200 import _native
from helpers import record_margin
from oracle import switchwhiten_oracle as so

DEV = torch.device("cuda:0")
RTOL = 2e-5

# ------------------------------------------------------------------------------------ the planner restated
NUM_SMS, CTAS_PER_SM, MOM_THREADS, MIN_CHUNK = 148, 2, 128, 512
FWD_STAGES, BWD_STAGES = 8, 6
BWD_ROWS = 8


def cdiv(a, b):
    return -(-a // b)


def plan_split(ng, hw, z):
    """sw_kernels.cu: plan_split, plus which limit set the split count and what the CTAs run."""
    budget = NUM_SMS * CTAS_PER_SM // (ng * z)
    most = cdiv(hw, MIN_CHUNK)
    if budget < 1:
        want, limit = 1, "clamp"
    elif budget > most:
        want, limit = most, "most"
    else:
        want, limit = budget, "budget"
    chunk = cdiv(cdiv(hw, want), MOM_THREADS) * MOM_THREADS
    splits = cdiv(hw, chunk)
    return {"limit": limit, "chunk": chunk, "splits": splits, "iters": cdiv(min(chunk, hw), MOM_THREADS),
            "last": hw - (splits - 1) * chunk}


def bwd_z(cp):
    return cp // min(cp, BWD_ROWS)


def arm_tags(shape):
    n, ch, h, w, cp = shape
    ng, hw = n * (ch // cp), h * w
    tags = set()
    for name, z, stages in (("fwd", 1, FWD_STAGES), ("bwd", bwd_z(cp), BWD_STAGES)):
        p = plan_split(ng, hw, z)
        tags.add(f"{name}:{p['limit']}")
        it = p["iters"]
        tags.update({stages - 1: {f"{name}:iters=S-1"}, stages: {f"{name}:iters=S"},
                     stages + 1: {f"{name}:iters=S+1"}}.get(it, set()))
        if it >= 3 * stages:
            tags.add(f"{name}:wraps>=3")
        if p["splits"] > 1:
            if p["last"] == 1:
                tags.add(f"{name}:last=1")
            elif p["last"] < MOM_THREADS:
                tags.add(f"{name}:last<128")
            elif p["last"] == p["chunk"]:
                tags.add(f"{name}:last=full")
    if hw == 1:
        tags.add("hw=1")
    elif hw == 2:
        tags.add("hw=2")
    elif hw < MOM_THREADS:
        tags.add("hw<128")
    if hw > 512 and hw % 512 == 1:
        tags.add("hw%512=1")
    if hw % 512 == 511:
        tags.add("hw%512=511")
    return tags


def workspace_bytes(n, ch, hw, cp):
    """sw_kernels.cu: layout(); the partials region is sized by the two split plans."""
    ng, mat = n * (ch // cp), cp * cp
    fwd = ng * plan_split(ng, hw, 1)["splits"] * (cp + cp * (cp + 1) // 2 + cp) * 4
    bwd = ng * plan_split(ng, hw, bwd_z(cp))["splits"] * cp * (cp + 1) * 4
    sizes = [max(fwd, bwd), ng * mat * 8, n * ch * 8, ng * 10 * 8, n * 4 * 8, n * ch * 8, n * ch * 8, n * ch * 4,
             ng * mat * 4, ng * mat * 4, n * ch * 4]
    o = 0
    for s in sizes:
        o = cdiv(o + s, 256) * 256
    return o


# ------------------------------------------------------------------------------------ cases
def mode(sw_type, tie=False, affine=True, training=True, T=5):
    return {"sw_type": sw_type, "tie": tie, "affine": affine, "training": training, "T": T}


PLAN_CASES = {  # id: ((n, ch, h, w, cp), mode, arms the shape was built to reach)
    "clamp-ring8-cp4": ((2, 600, 32, 32, 4), mode(2), {"fwd:clamp", "fwd:iters=S", "bwd:clamp"}),
    "clamp-wraps-cp16": ((10, 480, 48, 48, 16), mode(5), {"fwd:clamp", "bwd:clamp", "bwd:wraps>=3"}),
    "last1-cp16": ((2, 592, 29, 53, 16), mode(3, tie=True, T=8),
                   {"fwd:budget", "fwd:last=1", "bwd:budget", "bwd:iters=S+1", "hw%512=1"}),
    "clamp-wraps-cp4": ((3, 400, 40, 80, 4), mode(3, affine=False, T=1),
                        {"fwd:clamp", "fwd:wraps>=3", "bwd:clamp", "bwd:wraps>=3"}),
    "iters7-cp8": ((2, 600, 28, 28, 8), mode(2, training=False), {"fwd:budget", "fwd:iters=S-1", "bwd:iters=S+1"}),
    "iters9-cp16": ((2, 1200, 32, 33, 16), mode(2), {"fwd:budget", "fwd:iters=S+1", "bwd:clamp"}),
    "bwd-iters5-cp16": ((3, 400, 74, 7, 16), mode(5, tie=True, affine=False, training=False, T=8),
                        {"fwd:most", "bwd:budget", "bwd:iters=S-1"}),
    "bwd-iters6-cp16": ((3, 400, 92, 7, 16), mode(3), {"bwd:budget", "bwd:iters=S"}),
    "budget-wraps-cp8": ((3, 264, 77, 77, 8), mode(5), {"fwd:budget", "fwd:wraps>=3", "bwd:budget", "bwd:wraps>=3"}),
    "full-splits-cp4": ((1, 592, 80, 80, 4), mode(5, tie=True, training=False),
                        {"fwd:last=full", "fwd:wraps>=3", "bwd:last=full", "bwd:wraps>=3"}),
    "last-lt128-cp8": ((2, 8, 39, 40, 8), mode(3, tie=True, T=1), {"fwd:most", "fwd:last<128", "bwd:most", "bwd:last<128"}),
    "bwd-last1-cp16": ((2, 16, 29, 53, 16), mode(2, affine=False), {"fwd:most", "bwd:most", "bwd:last=1", "hw%512=1"}),
    "hw4095-cp8": ((2, 8, 45, 91, 8), mode(2, tie=True, training=False, T=8), {"hw%512=511"}),
    "hw511-cp4": ((3, 12, 73, 7, 4), mode(5, T=8), {"fwd:most", "hw%512=511"}),
    "hw99-cp8": ((3, 32, 9, 11, 8), mode(5), {"hw<128"}),
    "hw2-cp16": ((4, 32, 1, 2, 16), mode(3), {"hw=2"}),
    "hw1-cp4": ((3, 16, 1, 1, 4), mode(2), {"hw=1"}),
}

REQUIRED_ARMS = {f"{p}:{a}" for p in ("fwd", "bwd") for a in ("budget", "most", "clamp", "iters=S-1", "iters=S",
                                                               "iters=S+1", "wraps>=3", "last=1", "last<128", "last=full")}
REQUIRED_ARMS |= {"hw=1", "hw=2", "hw<128", "hw%512=1", "hw%512=511"}

OFFSET_SHAPES = {  # a multi-split plane and a one-split plane (n * groups > 296)
    "multi": ((2, 64, 40, 40, 16), mode(2), {"fwd:most", "bwd:most"}),
    "one": ((3, 400, 40, 80, 4), mode(3), {"fwd:clamp", "bwd:clamp", "fwd:wraps>=3"}),
}
OFFSETS = ["pixel0-10sd", "pixel0-30sd", "pixel0-100sd", "constant-but-pixel0", "mean-10sd", "mean-100sd"]


def make_inputs(shape, md, seed, offset=None):
    n, ch, h, w, cp = shape
    g = torch.Generator().manual_seed(seed)
    scale = 0.5 + torch.rand(1, ch, 1, 1, generator=g)
    x = torch.randn(n, ch, h, w, generator=g) * scale + 0.8 * torch.randn(1, ch, 1, 1, generator=g)
    x = x + 0.4 * x.roll(1, dims=1)
    if offset is not None:
        x64 = x.double()
        sd = x64.reshape(n, ch, -1).std(-1).clamp_min(1e-3)     # per (sample, channel)
        if offset.startswith("pixel0"):
            k = float(offset.split("-")[1][:-2])
            x64[:, :cp, 0, 0] += k * sd[:, :cp]
        elif offset == "constant-but-pixel0":
            x64[:, :cp] = x64[:, :cp, :1, :1]
            x64[:, :cp, 0, 0] += 3.0 * sd[:, :cp]
        else:
            k = float(offset.split("-")[1][:-2])
            x64 += k * sd.mean(0)[None, :, None, None]
        x = x64.float()
    a = torch.randn(ch // cp, cp, cp, generator=g)
    return {
        "x": x, "gy": torch.randn(n, ch, h, w, generator=g),
        "mw": torch.randn(md["sw_type"], generator=g),
        "vw": None if md["tie"] else torch.randn(md["sw_type"], generator=g),
        "weight": 1 + 0.3 * torch.randn(ch, generator=g) if md["affine"] else None,
        "bias": 0.3 * torch.randn(ch, generator=g) if md["affine"] else None,
        "rmean": 0.3 * torch.randn(ch // cp, cp, 1, generator=g),
        "rcov": a @ a.transpose(1, 2) / cp + 0.2 * torch.eye(cp),
    }


# ------------------------------------------------------------------------------------ checks on the host
ALL_SHAPES = {**{k: (v[0], v[2]) for k, v in PLAN_CASES.items()}, **{f"offset-{k}": (v[0], v[2]) for k, v in OFFSET_SHAPES.items()}}


@pytest.mark.parametrize("name", list(ALL_SHAPES))
def test_case_lands_on_its_arms(name):
    shape, want = ALL_SHAPES[name]
    got = arm_tags(shape)
    assert want <= got, f"{name} {shape}: misses {sorted(want - got)}; the planner puts it on {sorted(got)}"
    n, ch, h, w, _ = shape
    assert n * ch * h * w * 4 <= 50e6, "keep the file fast: inputs under 50 MB"


def test_cases_cover_every_arm_and_mode():
    covered = set().union(*(t for _, _, t in PLAN_CASES.values()))
    assert REQUIRED_ARMS <= covered, sorted(REQUIRED_ARMS - covered)
    assert any(s[4] == 16 and "bwd:wraps>=3" in t and "bwd:clamp" in t for s, _, t in PLAN_CASES.values())  # z = 2
    modes = [(s[4], m) for s, m, _ in PLAN_CASES.values()]
    assert {(cp, m["sw_type"]) for cp, m in modes} == {(cp, t) for cp in (4, 8, 16) for t in (2, 3, 5)}
    assert {cp for cp, m in modes if m["training"]} == {4, 8, 16}
    for key, values in (("tie", {True, False}), ("affine", {True, False}), ("training", {True, False}), ("T", {1, 5, 8})):
        assert {m[key] for _, m in modes} == values, key


def test_planner_restatement_matches_the_library():
    """The workspace the library asks for is laid out from its two split plans: equal sizes for every case and for a
    sweep of shapes mean the restated planner splits like the real one."""
    lib = _native.lib()
    shapes = [s for s, _ in ALL_SHAPES.values()]
    rng = np.random.default_rng(7)
    for _ in range(400):
        cp = int(rng.choice([4, 8, 16]))
        shapes.append((int(rng.integers(1, 17)), cp * int(rng.integers(1, 80)), int(rng.integers(1, 200)),
                       int(rng.integers(1, 200)), cp))
    for n, ch, h, w, cp in shapes:
        assert lib.dgvcc_sw_workspace_bytes(n, ch, h * w, cp) == workspace_bytes(n, ch, h * w, cp), (n, ch, h, w, cp)


def test_oracle_shift_is_a_sample_mean():
    """``decomposed`` centres the moments where the kernel does: on the fp32 mean of pixels (t // 8) hw // 16 + t % 8."""
    xg = np.arange(2 * 3 * 1000, dtype=np.float64).reshape(1, 2, 3, 1000) ** 1.5
    idx = [((t >> 3) * 1000) // 16 + (t & 7) for t in range(128)]
    assert len(set(idx)) == 128 and max(idx) < 1000
    assert np.array_equal(so.sample_shift(xg), xg[..., idx].mean(-1).astype(np.float32).astype(np.float64))
    small = np.random.default_rng(0).standard_normal((1, 1, 2, 77))
    assert np.array_equal(so.sample_shift(small), small.mean(-1).astype(np.float32).astype(np.float64))


# ------------------------------------------------------------------------------------ the C entry points, one by one
def stages_via_abi(inp, shape, md):
    """The module's sequence of C calls (models/ISW/switchwhiten.py), every output kept; workspace filled with NaN."""
    n, ch, h, w, cp = shape
    hw, groups = h * w, ch // cp
    lib, st, ptr = _native.lib(), _native.stream_ptr(DEV), _native.ptr
    dev = lambda t: None if t is None else t.to(DEV).contiguous()
    x, gy, mw, vw, wt, bs = (dev(inp[k]) for k in ("x", "gy", "mw", "vw", "weight", "bias"))
    nbytes = lib.dgvcc_sw_workspace_bytes(n, ch, hw, cp)
    ws = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device=DEV)      # every float and double in it is NaN
    f64 = lambda *s: torch.full(s, float("nan"), dtype=torch.float64, device=DEV)
    out = {"mean_in": f64(n, ch), "cov_in": f64(n, groups, cp, cp)}
    _native.check(lib.dgvcc_sw_instance_stats(ptr(x), n, ch, hw, cp, ptr(out["mean_in"]), ptr(out["cov_in"]), ptr(ws),
                                              nbytes, st), "instance_stats")
    rmean, rcov = dev(inp["rmean"]).clone(), dev(inp["rcov"]).clone()
    if md["training"]:
        out["mean_bn"], out["cov_bn"] = f64(ch), f64(groups, cp, cp)
        _native.check(lib.dgvcc_sw_batch_mean(ptr(out["mean_in"]), n, ch, ptr(out["mean_bn"]), st), "batch_mean")
        _native.check(lib.dgvcc_sw_batch_cov(ptr(out["mean_in"]), ptr(out["cov_in"]), ptr(out["mean_bn"]), n, ch, cp,
                                             ptr(out["cov_bn"]), st), "batch_cov")
        _native.check(lib.dgvcc_sw_update_running(ptr(rmean), ptr(rcov), ptr(out["mean_bn"]), ptr(out["cov_bn"]), ch, cp,
                                                  0.99, 1 - 0.99, st), "update_running")
        bn_scale = 1.0 / (n * hw)
    else:
        out["mean_bn"], out["cov_bn"] = rmean.double().reshape(ch).contiguous(), rcov.double().contiguous()
        bn_scale = 0.0
    out["rmean"], out["rcov"] = rmean, rcov
    out["a_fwd"] = torch.full((n, groups, cp, cp), float("nan"), device=DEV)
    out["y"] = torch.full_like(x, float("nan"))
    _native.check(lib.dgvcc_sw_whiten_forward(ptr(x), ptr(out["mean_in"]), ptr(out["cov_in"]), ptr(out["mean_bn"]),
                                              ptr(out["cov_bn"]), ptr(mw), ptr(vw), ptr(wt), ptr(bs), n, ch, hw, cp,
                                              md["sw_type"], md["T"], 1e-5, ptr(out["a_fwd"]), ptr(out["y"]), ptr(ws),
                                              nbytes, st), "whiten_forward")
    nan32 = lambda t: None if t is None else torch.full_like(t, float("nan"))
    out["gmw"], out["gvw"], out["gweight"], out["gbias"] = nan32(mw), nan32(vw), nan32(wt), nan32(bs)
    out["g_mean_bn"], out["g_cov_bn"] = f64(ch), f64(groups, cp, cp)
    _native.check(lib.dgvcc_sw_backward_stats(ptr(x), ptr(gy), ptr(out["mean_in"]), ptr(out["cov_in"]), ptr(out["mean_bn"]),
                                              ptr(out["cov_bn"]), ptr(mw), ptr(vw), ptr(wt), n, ch, hw, cp, md["sw_type"],
                                              md["T"], 1e-5, ptr(out["gmw"]), ptr(out["gvw"]), ptr(out["gweight"]),
                                              ptr(out["gbias"]), ptr(out["g_mean_bn"]), ptr(out["g_cov_bn"]), ptr(ws),
                                              nbytes, st), "backward_stats")
    out["gx"] = torch.full_like(x, float("nan"))
    _native.check(lib.dgvcc_sw_backward_apply(ptr(x), ptr(gy), ptr(out["a_fwd"]), ptr(out["mean_in"]), ptr(out["mean_bn"]),
                                              ptr(out["g_mean_bn"]), ptr(out["g_cov_bn"]), ptr(mw), ptr(vw), bn_scale, n,
                                              ch, hw, cp, md["sw_type"], ptr(out["gx"]), ptr(ws), nbytes, st),
                  "backward_apply")
    torch.cuda.synchronize()
    return {k: None if v is None else v.cpu() for k, v in out.items()}


def run_module(inp, shape, md):
    from dgvcc_b200.models.ISW.switchwhiten import SwitchWhiten2d
    m = SwitchWhiten2d(shape[1], num_pergroup=shape[4], sw_type=md["sw_type"], T=md["T"], tie_weight=md["tie"],
                       affine=md["affine"]).to(DEV)
    with torch.no_grad():
        m.sw_mean_weight.copy_(inp["mw"])
        if not md["tie"]:
            m.sw_var_weight.copy_(inp["vw"])
        if md["affine"]:
            m.weight.copy_(inp["weight"])
            m.bias.copy_(inp["bias"])
        m.running_mean.copy_(inp["rmean"])
        m.running_cov.copy_(inp["rcov"])
    m.train(md["training"])
    x = inp["x"].to(DEV).requires_grad_(True)
    y = m(x)
    y.backward(inp["gy"].to(DEV))
    torch.cuda.synchronize()
    out = {"y": y.detach(), "gx": x.grad, "gmw": m.sw_mean_weight.grad, "rmean": m.running_mean, "rcov": m.running_cov,
           "gvw": None if md["tie"] else m.sw_var_weight.grad}
    out["gweight"], out["gbias"] = (m.weight.grad, m.bias.grad) if md["affine"] else (None, None)
    return {k: None if v is None else v.detach().cpu() for k, v in out.items()}


def gate(got, ref, what, block=None):
    """|got - ref| <= RTOL (|ref| + max|ref|), the max over the trailing ``block`` dimensions when given."""
    got = torch.as_tensor(np.asarray(got, np.float64)).reshape(np.shape(ref))
    ref = torch.as_tensor(np.asarray(ref, np.float64))
    scale = ref.abs()
    if block:
        peak = scale.reshape(*scale.shape[:-block], -1).max(-1).values.reshape(*scale.shape[:-block], *([1] * block))
    else:
        peak = scale.max()
    tol = RTOL * (scale + peak)
    err = (got - ref).abs()
    err = torch.where(torch.isnan(err), torch.full_like(err, float("inf")), err)
    record_margin(what, err, tol, RTOL, 0.0)
    bad = err > tol
    if bad.any():
        idx = tuple(torch.nonzero(bad)[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())}/{bad.numel()} outside the gate, worst err/gate "
                             f"{float((err / tol.clamp_min(1e-300)).max()):.3g}; first at {idx}: got {float(got[idx]):.9g} "
                             f"ref {float(ref[idx]):.9g}")


def accuracy(got, ref, what):
    got = torch.as_tensor(np.asarray(got, np.float64)).reshape(np.shape(ref))
    ref = torch.as_tensor(np.asarray(ref, np.float64))
    record_margin(f"{what} (accuracy)", (got - ref).abs(), RTOL * (ref.abs() + ref.abs().max()), RTOL, 0.0)


GRADS = {"gx": "x", "gmw": "sw_mean_weight", "gvw": "sw_var_weight", "gweight": "weight", "gbias": "bias"}


def check_against_fp64(inp, shape, md):
    n, ch, h, w, cp = shape
    groups = ch // cp
    opt = lambda t: None if t is None else t.numpy()
    st64 = {}
    y64, g64, (mean_bn64, cov_bn64) = so.decomposed(
        inp["x"].numpy(), inp["gy"].numpy(), opt(inp["mw"]), opt(inp["vw"]), opt(inp["weight"]), opt(inp["bias"]),
        inp["rmean"].numpy(), inp["rcov"].numpy(), num_pergroup=cp, sw_type=md["sw_type"], T=md["T"],
        training=md["training"], stages=st64)
    got = stages_via_abi(inp, shape, md)

    # instance statistics against two-pass fp64 statistics of the fp32 input (not the shifted restatement)
    xg = inp["x"].double().reshape(n, groups, cp, -1)
    mean2 = xg.mean(-1)
    xc = xg - mean2[..., None]
    cov2 = xc @ xc.transpose(-1, -2) / xg.shape[-1]
    gate(got["mean_in"].reshape(n, groups, cp), mean2, "mean_in", block=1)
    gate(got["cov_in"], cov2, "cov_in", block=2)
    if md["training"]:
        gate(got["mean_bn"].reshape(groups, cp), mean_bn64, "batch_mean")
        gate(got["cov_bn"], cov_bn64, "batch_cov")
        rm = inp["rmean"].double() * 0.99 + 0.01 * torch.from_numpy(mean_bn64)[..., None]
        rc = inp["rcov"].double() * 0.99 + 0.01 * torch.from_numpy(cov_bn64)
    else:
        rm, rc = inp["rmean"].double(), inp["rcov"].double()
    gate(got["rmean"], rm, "running_mean")
    gate(got["rcov"], rc, "running_cov")
    gate(got["a_fwd"], st64["a_fwd"], "a_fwd", block=2)
    gate(got["y"], y64, "y")
    for k, leaf in GRADS.items():
        if g64[leaf] is not None:
            gate(got[k], g64[leaf], f"{k} ({'backward_apply' if k == 'gx' else 'backward_stats'})")
    gate(got["g_mean_bn"], st64["g_mean_bn"], "g_mean_bn")
    gate(got["g_cov_bn"], st64["g_cov_bn"], "g_cov_bn")

    # the module issues the same launches: the same bits
    mod = run_module(inp, shape, md)
    for k in ("y", "gx", "gmw", "gvw", "gweight", "gbias", "rmean", "rcov"):
        assert (mod[k] is None) == (got[k] is None), k
        if mod[k] is not None:
            assert torch.equal(mod[k].reshape(got[k].shape), got[k]), f"module {k} differs from the C entry points"

    # how far the reference's own fp32 evaluation sits from fp64, beside the kernels'
    rm32, rc32 = inp["rmean"].clone(), inp["rcov"].clone()
    y32, g32 = so.forward_backward(inp["x"], inp["gy"], inp["mw"], inp["vw"], inp["weight"], inp["bias"], rm32, rc32,
                                   num_pergroup=cp, sw_type=md["sw_type"], T=md["T"], training=md["training"])
    accuracy(y32.numpy(), y64, "fp32 reference y")
    accuracy(g32["x"].numpy(), g64["x"], "fp32 reference gx")
    accuracy(got["y"], y64, "kernel y")
    accuracy(got["gx"], g64["x"], "kernel gx")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PLAN_CASES))
def test_plan_arm_against_fp64(name):
    shape, md, _ = PLAN_CASES[name]
    seed = sum(shape) * 31 + md["sw_type"]
    check_against_fp64(make_inputs(shape, md, seed), shape, md)


@pytest.mark.gpu
@pytest.mark.parametrize("offset", OFFSETS)
@pytest.mark.parametrize("where", list(OFFSET_SHAPES))
def test_off_centre_plane_against_fp64(where, offset):
    shape, md, _ = OFFSET_SHAPES[where]
    check_against_fp64(make_inputs(shape, md, 1000 + OFFSETS.index(offset), offset), shape, md)


@pytest.mark.gpu
def test_one_split_wrap_shape_is_bit_reproducible():
    """The one-split shape whose backward ring wraps three times: two forward + backward passes, the same bits."""
    shape, md, _ = PLAN_CASES["clamp-wraps-cp16"]
    inp = make_inputs(shape, md, 99)
    a, b = run_module(inp, shape, md), run_module(inp, shape, md)
    for k, v in a.items():
        if v is not None:
            assert torch.equal(v, b[k]), k
