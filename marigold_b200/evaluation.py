"""Device-side evaluation step that follows the hot path in dataset evaluation (csrc/eval.cu), one host synchronisation
per sample:
  depth    least-squares scale / shift alignment in depth or disparity (reference src/util/alignment.py:35-95,
           script/depth/eval.py:171-207) and the masked depth metrics of src/util/metric.py:64-191
  normals  compute_cosine_error(masked=True) and the angular metrics of src/util/metric.py:194-257
  iid      compute_iid_metric's PSNR (src/util/metric.py:263-338), with script/iid/eval.py:183-196's colour transforms"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr, stream_ptr

ALIGNMENTS = {None: 0, "least_square": 1, "least_square_disparity": 2}
NORMALS_METRIC_NAMES = ("mean_angular_error", "median_angular_error", "rmse_angular_error", "sub5_error", "sub7_5_error",
                        "sub11_25_error", "sub22_5_error", "sub30_error")
COLOR_TRANSFORMS = {None: 0, "srgb2linear": 1, "linear2srgb": 2}
METRIC_NAMES = ("abs_relative_difference", "squared_relative_difference", "rmse_linear", "rmse_log", "log10", "delta1_acc",
                "delta2_acc", "delta3_acc", "i_rmse", "silog_rmse")
_ws = {}


def _flat(pred, gt, mask):
    if not (pred.is_cuda and gt.is_cuda):
        raise _lib.MgbError("marigold_b200.evaluation needs CUDA tensors (no CPU fallback)")
    p = pred.to(torch.float32).contiguous().reshape(-1)
    g = gt.to(torch.float32).contiguous().reshape(-1)
    assert p.numel() == g.numel(), f"{tuple(pred.shape)} vs {tuple(gt.shape)}"
    m = None
    if mask is not None:
        m = mask.to(device=p.device).to(torch.uint8).contiguous().reshape(-1)
        assert m.numel() == p.numel()
    return p, g, m


def _workspace(lib, device):
    ws = _ws.get(device)
    if ws is None:
        ws = torch.empty(int(lib.mgb_eval_ws_bytes()), dtype=torch.uint8, device=device)
        _ws[device] = ws
    return ws


def _run(pred, gt, mask, alignment: int, dmin: float, dmax: float, want_aligned: bool):
    p, g, m = _flat(pred, gt, mask)
    lib = _lib.load()
    with torch.cuda.device(p.device):
        ws = _workspace(lib, p.device)
        aligned = torch.empty_like(p) if want_aligned else None
        out = np.zeros(13, dtype=np.float64)
        check(lib.mgb_eval_depth(ptr(p), ptr(g), ptr(m), p.numel(), int(alignment), float(dmin), float(dmax), ptr(aligned),
                                 ptr(ws), out.ctypes.data_as(C.c_void_p), stream_ptr()), "mgb_eval_depth")
    return out, (aligned.reshape(pred.shape) if aligned is not None else None)


def align_depth_least_square(gt: torch.Tensor, pred: torch.Tensor, valid_mask: Optional[torch.Tensor],
                             return_scale_shift: bool = True, max_resolution: Optional[int] = None):
    """src/util/alignment.py:35-82 on the device: (aligned_pred, scale, shift). `max_resolution` downsamples the three
    maps with the reference's nearest Upsample before the fit; the fitted map is always the full-resolution prediction."""
    fit_p, fit_g, fit_m = pred, gt, valid_mask
    if max_resolution is not None:
        sf = float(np.min(max_resolution / np.array(pred.shape[-2:])))
        if sf < 1:
            down = torch.nn.Upsample(scale_factor=sf, mode="nearest")
            fit_g = down(gt.reshape(1, 1, *gt.shape[-2:]).float())
            fit_p = down(pred.reshape(1, 1, *pred.shape[-2:]).float())
            fit_m = down(valid_mask.reshape(1, 1, *valid_mask.shape[-2:]).float()).bool() if valid_mask is not None else None
    out, _ = _run(fit_p, fit_g, fit_m, 1, -3.0e38, 3.0e38, False)      # only the fit is used from this call
    scale, shift = out[0], out[1]
    aligned = pred.to(torch.float64) * scale + shift
    return (aligned, scale, shift) if return_scale_shift else aligned


def evaluate_depth(pred: torch.Tensor, gt: torch.Tensor, valid_mask: Optional[torch.Tensor] = None,
                   alignment: Optional[str] = "least_square", min_depth: float = 1e-6, max_depth: float = 3.0e38,
                   return_aligned: bool = False):
    """One sample of script/depth/eval.py:171-217: align (or not), clip to the dataset range and to d > 1e-6, all metrics.
    alignment: None, "least_square" (in depth) or "least_square_disparity" (pred fitted to 1 / gt over the valid pixels
    with gt > 0 and pred > 0, depth = 1 / clip(pred * scale + shift, 1e-3)).
    Returns (metrics by the reference's function names, {"scale", "shift", "n_valid"}), plus the final depth map the
    metrics were computed on when return_aligned; scale and shift are in disparity space for "least_square_disparity"."""
    if alignment not in ALIGNMENTS:
        raise ValueError(f"unsupported alignment {alignment!r}; expected one of {list(ALIGNMENTS)}")
    out, aligned = _run(pred, gt, valid_mask, ALIGNMENTS[alignment], min_depth, max_depth, return_aligned)
    metrics = dict(zip(METRIC_NAMES, (float(v) for v in out[3:13])))
    info = {"scale": float(out[0]), "shift": float(out[1]), "n_valid": int(out[2])}
    return (metrics, info, aligned) if return_aligned else (metrics, info)


def _chw(x: torch.Tensor, what: str) -> torch.Tensor:
    if x.dim() == 4 and x.shape[0] == 1:
        x = x[0]
    if x.dim() != 3 or x.shape[0] != 3:
        raise ValueError(f"{what}: expected [3,H,W] or [1,3,H,W], got {tuple(x.shape)}")
    return x


def evaluate_normals(pred: torch.Tensor, gt: torch.Tensor, return_errors: bool = False):
    """One sample of script/normals/eval.py:145-157: compute_cosine_error(pred, gt, masked=True) and the metric functions
    of src/util/metric.py:222-257 (rounded with their round(., 4)); pixels with a zero ground-truth vector are left out.
    The median is an exact order statistic computed on the device. pred, gt: [3,H,W] or [1,3,H,W].
    Returns (metrics by the reference's function names, {"n_valid"}), plus the [H,W] angular error map in degrees (NaN
    where the ground truth is zero) when return_errors. Metrics are NaN when no pixel is valid."""
    out, angles = normals_raw(pred, gt, return_errors)
    # the reference rounds mean / median / rmse as numpy float32 scalars and the percentages as float64
    metrics = {k: float(round(np.float32(v), 4)) if i < 3 else round(float(v), 4)
               for i, (k, v) in enumerate(zip(NORMALS_METRIC_NAMES, out[1:9]))}
    info = {"n_valid": int(out[0])}
    return (metrics, info, angles) if return_errors else (metrics, info)


def normals_raw(pred: torch.Tensor, gt: torch.Tensor, return_errors: bool = False):
    """evaluate_normals before rounding: (float64 [9] = {n_valid, mean, median, rmse, % < 5, 7.5, 11.25, 22.5, 30},
    [H,W] angle map or None). The median is the float32 value np.median returns."""
    pred, gt = _chw(pred, "pred"), _chw(gt, "gt")
    assert pred.shape == gt.shape, f"{tuple(pred.shape)} vs {tuple(gt.shape)}"
    p, g, _ = _flat(pred, gt, None)
    lib = _lib.load()
    HW = gt.shape[1] * gt.shape[2]
    with torch.cuda.device(p.device):
        ws = _workspace(lib, p.device)
        angles = torch.empty(HW, dtype=torch.float32, device=p.device) if return_errors else None
        out = np.zeros(9, dtype=np.float64)
        check(lib.mgb_eval_normals(ptr(p), ptr(g), HW, ptr(angles), ptr(ws), out.ctypes.data_as(C.c_void_p), stream_ptr()),
              "mgb_eval_normals")
    return out, (angles.reshape(gt.shape[1:]) if angles is not None else None)


def evaluate_iid(pred: torch.Tensor, gt: torch.Tensor, target_name: str, valid_mask: Optional[torch.Tensor] = None,
                 color_transform: Optional[str] = None):
    """One target of one sample of script/iid/eval.py:182-213 for the PSNR metric: the optional colour transform
    ("srgb2linear": x ** 2.2, "linear2srgb": x ** (1 / 2.2), applied to both), then compute_iid_metric: for "shading" and
    "residual" a least-squares scale and quantile_map (the gt brightness' 0.9 quantile is an exact order statistic on the
    device), and PSNR(data_range=1) over the masked elements. pred, gt and valid_mask (per channel): [3,H,W] or [1,3,H,W].
    Returns ({"psnr"}, {"lstsq_scale", "quantile", "quantile_scale", "n"}); the alignment values are NaN for targets that
    are not aligned."""
    if color_transform not in COLOR_TRANSFORMS:
        raise ValueError(f"unsupported color_transform {color_transform!r}; expected one of {list(COLOR_TRANSFORMS)}")
    pred, gt = _chw(pred, "pred"), _chw(gt, "gt")
    assert pred.shape == gt.shape, f"{tuple(pred.shape)} vs {tuple(gt.shape)}"
    if valid_mask is not None:
        valid_mask = _chw(valid_mask, "valid_mask")
    p, g, m = _flat(pred, gt, valid_mask)
    lib = _lib.load()
    HW = gt.shape[1] * gt.shape[2]
    align = target_name in ("shading", "residual")
    with torch.cuda.device(p.device):
        ws = _workspace(lib, p.device)
        out = np.zeros(5, dtype=np.float64)
        check(lib.mgb_eval_iid(ptr(p), ptr(g), ptr(m), HW, int(align), COLOR_TRANSFORMS[color_transform], ptr(ws),
                               out.ctypes.data_as(C.c_void_p), stream_ptr()), "mgb_eval_iid")
    return {"psnr": float(out[0])}, {"lstsq_scale": float(out[1]), "quantile": float(out[2]),
                                     "quantile_scale": float(out[3]), "n": int(out[4])}
