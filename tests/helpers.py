"""Shared helpers for the parity tests."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_bl_golden(name):
    z = np.load(os.path.join(GOLDEN, f"bl_{name}.npz"))
    B = len(z["in_counts"])
    case = {
        "width": int(z["in_width"]), "height": int(z["in_height"]), "stride": int(z["in_stride"]),
        "sigma": float(z["in_sigma"]), "use_bg": bool(int(z["in_use_bg"])), "bg_ratio": float(z["in_bg_ratio"]),
        "st_sizes": torch.from_numpy(z["in_st_sizes"].copy()),
        "density": torch.from_numpy(z["in_density"].copy()),
        "points": [torch.from_numpy(z[f"in_points_{i}"].copy()) for i in range(B)],
        "targets": [torch.from_numpy(z[f"in_targets_{i}"].copy()) for i in range(B)],
        "ref_loss": torch.from_numpy(z["ref_loss"].copy()),
        "ref_grad": torch.from_numpy(z["ref_grad"].copy()),
        "ref_count": {}, "ref_colsum": {}, "ref_prob_rows": {}, "ref_prob": {},
    }
    for i in range(B):
        if f"ref_count_{i}" in z:
            case["ref_count"][i] = torch.from_numpy(z[f"ref_count_{i}"].copy())
            case["ref_colsum"][i] = torch.from_numpy(z[f"ref_colsum_{i}"].copy())
            case["ref_prob_rows"][i] = z[f"ref_prob_rows_{i}"].tolist()
            case["ref_prob"][i] = torch.from_numpy(z[f"ref_prob_{i}"].copy())
    return case


BL_GOLDEN_CASES = ["c1", "mixed", "nobg", "empty", "sigma10", "outside"]


# (test id, what, worst err / gate, rtol, atol) of every tolerance check that ran: conftest.py prints the worst one
# per test at the end of the session, so the log shows how far inside its gate each parity test sits.
MARGINS = []


def record_margin(what, err, tol, rtol, atol):
    """err, tol: float64 tensors of equal shape (|got - ref| and atol + rtol |ref|)."""
    if err.numel() == 0:
        return
    ratio = torch.where(tol > 0, err / tol.clamp_min(1e-300), torch.where(err > 0, torch.inf, 0.0).to(err.dtype))
    test = os.environ.get("PYTEST_CURRENT_TEST", "?").split(" (")[0]
    MARGINS.append((test, what, float(ratio.max()), float(rtol), float(atol)))


def assert_close(got, ref, rtol, atol, what=""):
    got = torch.as_tensor(got).double()
    ref = torch.as_tensor(ref).double()
    err = (got - ref).abs()
    tol = atol + rtol * ref.abs()
    record_margin(what, err, tol, rtol, atol)
    bad = err > tol
    if bad.any():
        idx = torch.nonzero(bad)[0].tolist()
        worst = (err / tol).max().item()
        raise AssertionError(
            f"{what}: {int(bad.sum())}/{bad.numel()} out of tolerance (rtol={rtol}, atol={atol}); "
            f"worst err/tol={worst:.3g}; first at {idx}: got {got[tuple(idx)].item():.9g} ref {ref[tuple(idx)].item():.9g}")


def load_sw_cases():
    """tests/golden/sw_cases.npz -> {name: dict(cfg..., inputs as torch tensors, ref outputs per rank)}."""
    z = np.load(os.path.join(GOLDEN, "sw_cases.npz"))
    cases = {}
    for key in z.files:
        if key.startswith("in_") and key.endswith("_cfg"):
            name = key[3:-4]
            cper, sw_type, tie, affine, training, kind = (int(v) for v in z[key])
            c = {"num_pergroup": cper, "sw_type": sw_type, "tie": bool(tie), "affine": bool(affine),
                 "training": bool(training), "kind": ("plain", "sync1", "sync2")[kind]}
            for k in ("x", "gy", "mw", "vw", "weight", "bias", "rmean", "rcov"):
                c[k] = torch.from_numpy(z[f"in_{name}_{k}"].copy()) if f"in_{name}_{k}" in z.files else None
            world = 2 if c["kind"] == "sync2" else 1
            prefix = [f"ref_{name}_"] if c["kind"] == "plain" else [f"ref_{name}_r{r}_" for r in range(world)]
            c["world"] = world
            c["ref"] = [{k[len(p):]: z[k] for k in z.files if k.startswith(p)} for p in prefix]
            cases[name] = c
    return cases


def assert_map_close(got, ref, what):
    """Density-map gate (SURVEY.md section 8d): rtol 1e-5 with atol 1e-7*max|ref|; returns the number of pixels that are
    not bit-identical."""
    assert got.dtype == np.float32 and got.shape == ref.shape
    tol = 1e-5 * np.abs(ref) + 1e-7 * float(np.abs(ref).max() if ref.size else 0)
    bad = np.abs(got.astype(np.float64) - ref) > tol
    assert not bad.any(), f"{what}: {int(bad.sum())} pixels out of tolerance, max err {np.abs(got - ref).max()}"
    return int((got != ref).sum())
