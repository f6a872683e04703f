"""REFERENCE RESTATEMENT (test infrastructure only; never imported by the product path).

Plain torch / numpy restatement of the reference's evaluation code for the modes marigold_b200.evaluation adds:
  depth, least_square_disparity  script/depth/eval.py:179-217 with align_depth_least_square and depth2disparity
                                 (src/util/alignment.py:35-95) and the depth metrics (src/util/metric.py:64-191)
  normals                        compute_cosine_error and the angular metric functions (src/util/metric.py:194-257)
  iid                            compute_alignment_scale, quantile_map and compute_iid_metric's PSNR
                                 (src/util/metric.py:263-338), the colour transforms of script/iid/eval.py:183-196

Every function runs on the device of its inputs, so tools/eval_time.py times the reference's path with torch CUDA ops.
PARITY PINNED: tests/golden/eval_golden.npz holds what the reference's own functions returned on the inputs of
tests/golden/eval_cases.py (tests/golden/make_eval_golden.py); tests/test_eval_oracle.py checks this file against it.
"""
from __future__ import annotations

import numpy as np
import torch

DEPTH_METRICS = ("abs_relative_difference", "squared_relative_difference", "rmse_linear", "rmse_log", "log10",
                 "delta1_acc", "delta2_acc", "delta3_acc", "i_rmse", "silog_rmse")


# ---- depth, least_square_disparity ----------------------------------------------------------------------------------
def _lstsq_fit(gt: np.ndarray, pred: np.ndarray, mask: np.ndarray):
    g = gt[mask].reshape((-1, 1))
    p = pred[mask].reshape((-1, 1))
    X = np.linalg.lstsq(np.concatenate([p, np.ones_like(p)], axis=-1), g, rcond=None)[0]
    return X[0], X[1]


def _depth_metrics(o: torch.Tensor, t: torch.Tensor, m: torch.Tensor) -> dict:
    n = m.sum((-1, -2))

    def masked_mean(v):
        v = v.clone()
        v[~m] = 0
        return torch.sum(v, (-1, -2)) / n

    dl = torch.log(o) - torch.log(t)
    r = torch.max(o / t, t / o)

    def thr(x):
        b = torch.where(r.cpu() < x, torch.ones(*o.shape), torch.zeros(*o.shape))
        b[~m.cpu()] = 0
        return torch.sum(b, (-1, -2)) / n.cpu()

    return {
        "abs_relative_difference": masked_mean(torch.abs(o - t) / t),
        "squared_relative_difference": masked_mean(torch.pow(torch.abs(o - t), 2) / t),
        "rmse_linear": torch.sqrt(masked_mean(torch.pow(o - t, 2))),
        "rmse_log": torch.sqrt(masked_mean(torch.pow(dl, 2))),
        "log10": torch.abs(torch.log10(o[m]) - torch.log10(t[m])).mean(),
        "delta1_acc": thr(1.25), "delta2_acc": thr(1.25 ** 2), "delta3_acc": thr(1.25 ** 3),
        "i_rmse": torch.sqrt(masked_mean(torch.pow(1.0 / o - 1.0 / t, 2))),
        "silog_rmse": torch.sqrt(masked_mean(torch.pow(dl, 2)) - torch.pow(torch.sum(torch.where(m, dl, 0 * dl)), 2)
                                 / n ** 2) * 100,
    }


def eval_depth_disparity(pred: np.ndarray, gt: np.ndarray, mask: np.ndarray, dmin: float, dmax: float, device="cpu"):
    """script/depth/eval.py:179-217 for one sample. Returns (metrics, scale, shift, final depth)."""
    gt_disp = np.zeros_like(gt)
    gt_pos = gt > 0
    gt_disp[gt_pos] = 1.0 / gt[gt_pos]
    scale, shift = _lstsq_fit(gt_disp, pred, mask & gt_pos & (pred > 0))
    disp = np.clip(pred * scale + shift, a_min=1e-3, a_max=None)
    depth = np.zeros_like(disp)
    depth[disp > 0] = 1.0 / disp[disp > 0]
    depth = np.clip(np.clip(depth, a_min=dmin, a_max=dmax), a_min=1e-6, a_max=None)
    o = torch.from_numpy(depth).to(device)
    metrics = _depth_metrics(o, torch.from_numpy(gt).to(device), torch.from_numpy(mask).to(device))
    return {k: v.item() for k, v in metrics.items()}, float(scale[0]), float(shift[0]), depth


# ---- normals --------------------------------------------------------------------------------------------------------
def cosine_error(pred: torch.Tensor, gt: torch.Tensor) -> np.ndarray:
    """compute_cosine_error(pred, gt, masked=True): degrees over the pixels with ||gt|| > 0, flattened."""
    pred, gt = pred.reshape(3, -1), gt.reshape(3, -1)
    mask = torch.norm(gt, dim=0) > 0
    pred, gt = pred[:, mask], gt[:, mask]
    e = torch.clamp(torch.cosine_similarity(pred, gt, dim=0), min=-1.0, max=1.0)
    return (torch.acos(e) * 180.0 / np.pi).view(-1).detach().cpu().numpy()


def normals_metrics(err: np.ndarray) -> dict:
    n = err.shape[0]
    out = {"mean_angular_error": round(np.average(err), 4), "median_angular_error": round(np.median(err), 4),
           "rmse_angular_error": round(np.sqrt(np.sum(err * err) / n), 4)}
    for name, t in (("sub5_error", 5), ("sub7_5_error", 7.5), ("sub11_25_error", 11.25), ("sub22_5_error", 22.5),
                    ("sub30_error", 30)):
        out[name] = round(100.0 * (np.sum(err < t) / n), 4)
    return {k: float(v) for k, v in out.items()}


# ---- iid ------------------------------------------------------------------------------------------------------------
def srgb2linear(img):
    return img ** 2.2


def linear2srgb(img):
    return img ** (1.0 / 2.2)


def alignment_scale(pred, gt, valid_mask=None) -> torch.Tensor:
    pred, gt = pred.squeeze(), gt.squeeze()
    if valid_mask is not None:
        valid_mask = valid_mask.squeeze()
        pred, gt = pred[valid_mask], gt[valid_mask]
    return torch.linalg.lstsq(pred.reshape(-1, 1).float(), gt.reshape(-1, 1).float())[0]


def brightness(gt, valid_mask=None) -> torch.Tensor:
    gt = gt.squeeze()
    b = 0.3 * gt[0, :, :] + 0.59 * gt[1, :, :] + 0.11 * gt[2, :, :]
    return b[valid_mask.squeeze()[0]] if valid_mask is not None else b.flatten()


def quantile_map(pred, gt, valid_mask=None):
    """Returns (pred_mapped, gt_mapped, quantile, scale)."""
    q = torch.quantile(brightness(gt, valid_mask), 0.9)
    scale = 0 if q < 0.0001 else float(0.8 / q)
    pm = torch.clamp(scale * pred.squeeze(), 0, 1).unsqueeze(0)
    gm = torch.clamp(scale * gt.squeeze(), 0, 1).unsqueeze(0)
    return pm, gm, q, scale


def psnr(preds, target, data_range: float = 1.0):
    """torchmetrics' PeakSignalNoiseRatio(data_range=1.0) on one update."""
    diff = preds - target
    sse = torch.sum(diff * diff)
    n = torch.tensor(target.numel(), device=target.device)
    dr = torch.tensor(data_range, device=target.device)
    return (2 * torch.log(dr) - torch.log(sse / n)) * (10 / torch.log(torch.tensor(10.0)))


def eval_iid_psnr(pred, gt, target_name: str, valid_mask=None, color_transform=None) -> dict:
    """One target of script/iid/eval.py:182-213 with metric "psnr". pred, gt [1,3,H,W]; valid_mask [1,3,H,W] bool."""
    if color_transform == "srgb2linear":
        pred, gt = srgb2linear(pred), srgb2linear(gt)
    elif color_transform == "linear2srgb":
        pred, gt = linear2srgb(pred), linear2srgb(gt)
    info = {}
    if target_name in ("shading", "residual"):
        s = alignment_scale(pred, gt, valid_mask)
        pred = s * pred
        pred, gt, q, qs = quantile_map(pred, gt, valid_mask)
        info = {"lstsq_scale": s.item(), "quantile": q.item(), "quantile_scale": float(qs)}
    if valid_mask is not None:
        value = psnr(pred[valid_mask], gt[valid_mask]).item()
    else:
        value = psnr(pred, gt).item()
    return {"psnr": value, **info}
