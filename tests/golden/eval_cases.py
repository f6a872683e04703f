"""Seeded inputs of the evaluation goldens (tests/golden/eval_golden.npz), shared by make_eval_golden.py and the tests."""
import numpy as np
import torch

# least_square_disparity depth evaluation (script/depth/eval.py:179-217); dmin / dmax: the dataset's depth range
DISPARITY_CASES = {
    "d37x53_gt0_neg": dict(H=37, W=53, seed=61, gt_zero=40, neg_pred=30, dmin=1e-3, dmax=10.0),
    "d480x640": dict(H=480, W=640, seed=62, dmin=1e-3, dmax=10.0),
    "d480x640_neg": dict(H=480, W=640, seed=63, neg_pred=5000, dmin=0.5, dmax=8.0),
    "d37x53_nofit": dict(H=37, W=53, seed=64, all_negative=True, dmin=1e-3, dmax=10.0),
}
# normals (compute_cosine_error(masked=True) + metric.py:222-257); 37 x 53 = 1961 pixels, so zero_gt sets the parity
NORMALS_EVAL_CASES = {
    "n37x53_even": dict(H=37, W=53, seed=71, zero_gt=101, exact=60, anti=25, zero_pred=20),
    "n37x53_odd": dict(H=37, W=53, seed=72, zero_gt=100, exact=60, anti=25, zero_pred=20),
    "n480x640": dict(H=480, W=640, seed=73, zero_gt=15000, exact=2000, anti=500, zero_pred=300),
    "n480x640_odd": dict(H=480, W=640, seed=74, zero_gt=15001, exact=0, anti=0, zero_pred=0),
}
PIXEL_CASE = "n37x53_even"          # the one case whose per-pixel angles are stored
# IID PSNR (script/iid/eval.py:182-213 -> compute_iid_metric)
IID_EVAL_CASES = {
    "shading_mask": dict(H=37, W=53, seed=81, target="shading", mask=True),
    "shading_nomask_odd": dict(H=37, W=53, seed=82, target="shading", mask=False),
    "residual_mask": dict(H=37, W=53, seed=83, target="residual", mask=True),
    "albedo_mask": dict(H=37, W=53, seed=84, target="albedo", mask=True),
    "albedo_nomask": dict(H=37, W=53, seed=85, target="albedo", mask=False),
    "shading_dark": dict(H=37, W=53, seed=86, target="shading", mask=True, dark=True),
    "shading_srgb2linear": dict(H=37, W=53, seed=87, target="shading", mask=True, transform="srgb2linear"),
    "albedo_linear2srgb": dict(H=37, W=53, seed=88, target="albedo", mask=False, transform="linear2srgb"),
    "shading_768x1024": dict(H=768, W=1024, seed=89, target="shading", mask=True),
    "residual_768x1024": dict(H=768, W=1024, seed=90, target="residual", mask=False),
    "albedo_768x1024": dict(H=768, W=1024, seed=91, target="albedo", mask=True, transform="linear2srgb"),
}


def disparity_input(cfg):
    """(pred, gt, mask) float32 / float32 / bool [H,W]: gt depth in [0.5, 9.5], pred an affine map of the disparity plus
    noise (what an affine-invariant disparity model outputs)."""
    rng = np.random.default_rng(cfg["seed"])
    H, W = cfg["H"], cfg["W"]
    yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
    gt = (0.5 + 9.0 * (0.5 + 0.45 * np.sin(3 * xx + 2 * yy) * np.cos(2 * yy))).astype(np.float32)
    pred = (0.3 / gt + 0.05 + 0.002 * rng.standard_normal((H, W))).astype(np.float32)
    mask = rng.uniform(size=(H, W)) > 0.2
    idx = rng.permutation(H * W)
    if cfg.get("gt_zero"):
        sel = idx[: cfg["gt_zero"]]
        gt.reshape(-1)[sel] = 0.0
        mask.reshape(-1)[sel[: len(sel) // 2]] = True          # half of them inside the valid mask
    if cfg.get("neg_pred"):
        pred.reshape(-1)[idx[-cfg["neg_pred"]:]] *= -1.0
    if cfg.get("all_negative"):
        pred = -np.abs(pred)
    return pred, gt, mask


def normals_eval_input(cfg):
    """(pred, gt) float32 [3,H,W]: unit gt normals facing the camera, noisy unit predictions, and pixels with a zero gt
    vector, an exactly matching prediction, an antiparallel prediction and a zero prediction."""
    rng = np.random.default_rng(cfg["seed"])
    H, W = cfg["H"], cfg["W"]
    gt = rng.normal(size=(3, H, W))
    gt[2] += 2.0
    gt /= np.linalg.norm(gt, axis=0, keepdims=True)
    pred = gt + rng.normal(0, 0.25, size=(3, H, W))
    pred /= np.linalg.norm(pred, axis=0, keepdims=True)
    gt, pred = gt.astype(np.float32).reshape(3, -1), pred.astype(np.float32).reshape(3, -1)
    idx = rng.permutation(H * W)
    o = 0
    for key in ("zero_gt", "exact", "anti", "zero_pred"):
        sel = idx[o:o + cfg[key]]
        o += cfg[key]
        if key == "zero_gt":
            gt[:, sel] = 0.0
        elif key == "exact":
            pred[:, sel] = gt[:, sel]
        elif key == "anti":
            pred[:, sel] = -gt[:, sel]
        else:
            pred[:, sel] = 0.0
    return torch.from_numpy(pred.reshape(3, H, W)), torch.from_numpy(gt.reshape(3, H, W))


def iid_eval_input(cfg):
    """(pred, gt, mask or None): [1,3,H,W] float32 in [0,1] and a per-channel bool mask, as script/iid/eval.py loads
    them. Shading / residual predictions are off by a scale (they are up-to-scale targets)."""
    rng = np.random.default_rng(cfg["seed"])
    H, W = cfg["H"], cfg["W"]
    yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
    base = 0.5 + 0.35 * np.sin(4 * xx[None] + np.array([0.0, 1.0, 2.0])[:, None, None] + 3 * yy[None])
    gt = np.clip(base + 0.05 * rng.standard_normal((3, H, W)), 0, 1)
    if cfg.get("dark"):
        gt = gt * 5e-5
    k = 0.6 if cfg["target"] in ("shading", "residual") else 1.0
    pred = np.clip(k * gt + 0.04 * rng.standard_normal((3, H, W)), 0, 1)
    mask = torch.from_numpy(rng.uniform(size=(1, 3, H, W)) > 0.15) if cfg["mask"] else None
    return (torch.from_numpy(pred.astype(np.float32))[None], torch.from_numpy(gt.astype(np.float32))[None], mask)
