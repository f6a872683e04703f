"""Generate tests/golden/eval_golden.npz by running the REFERENCE's own evaluation code (needs /root/reference): the
metric and alignment functions of src/util/metric.py and src/util/alignment.py are imported live, and the glue of
script/depth/eval.py:179-217, script/normals/eval.py:145-157 and script/iid/eval.py:182-213 is restated around them
line for line. Inputs are regenerated from seeds by tests/golden/eval_cases.py, so only outputs are stored; per-pixel
arrays are kept for one small case of each task.

torchmetrics is not installed, so compute_iid_metric is called with a restated PSNR callable (torchmetrics'
PeakSignalNoiseRatio(data_range=1.0): 10 log10(1 / mse) in float32). Its masking, alignment scale and quantile map are
the reference's own code.

    python tests/golden/make_eval_golden.py
"""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from tests.golden._ref_eval_shim import load_reference_eval_utils  # noqa: E402
from tests.golden.eval_cases import (DISPARITY_CASES, IID_EVAL_CASES, NORMALS_EVAL_CASES, PIXEL_CASE,  # noqa: E402
                                     disparity_input, iid_eval_input, normals_eval_input)

ref = load_reference_eval_utils()
metric, alignment = ref["metric"], ref["alignment"]
out_dir = Path(__file__).resolve().parent
torch.set_num_threads(4)

DEPTH_FUNCS = [metric.abs_relative_difference, metric.squared_relative_difference, metric.rmse_linear, metric.rmse_log,
               metric.log10, metric.delta1_acc, metric.delta2_acc, metric.delta3_acc, metric.i_rmse, metric.silog_rmse]
NORMALS_FUNCS = [metric.mean_angular_error, metric.median_angular_error, metric.rmse_angular_error, metric.sub5_error,
                 metric.sub7_5_error, metric.sub11_25_error, metric.sub22_5_error, metric.sub30_error]


def psnr(preds, target):
    diff = preds - target
    sse = torch.sum(diff * diff)
    n = torch.tensor(target.numel())
    return (2 * torch.log(torch.tensor(1.0)) - torch.log(sse / n)) * (10 / torch.log(torch.tensor(10.0)))


store = {}
with np.errstate(divide="ignore", invalid="ignore"):
    for name, cfg in DISPARITY_CASES.items():
        depth_pred, depth_raw, valid_mask = disparity_input(cfg)
        # script/depth/eval.py:179-207
        gt_disparity, gt_non_neg_mask = alignment.depth2disparity(depth=depth_raw, return_mask=True)
        pred_non_neg_mask = depth_pred > 0
        valid_nonnegative_mask = valid_mask & gt_non_neg_mask & pred_non_neg_mask
        disparity_pred, scale, shift = alignment.align_depth_least_square(
            gt_arr=gt_disparity, pred_arr=depth_pred, valid_mask_arr=valid_nonnegative_mask, return_scale_shift=True,
            max_resolution=None)
        disparity_pred = np.clip(disparity_pred, a_min=1e-3, a_max=None)
        depth_pred = alignment.disparity2depth(disparity_pred)
        depth_pred = np.clip(depth_pred, a_min=cfg["dmin"], a_max=cfg["dmax"])
        depth_pred = np.clip(depth_pred, a_min=1e-6, a_max=None)
        # :209-217
        d_ts, g_ts, m_ts = torch.from_numpy(depth_pred), torch.from_numpy(depth_raw), torch.from_numpy(valid_mask)
        store[f"disp/{name}/metrics"] = np.array([f(d_ts, g_ts, m_ts).item() for f in DEPTH_FUNCS])
        store[f"disp/{name}/scale_shift"] = np.array([float(scale[0]), float(shift[0])])
        store[f"disp/{name}/n_fit"] = np.array(int(valid_nonnegative_mask.sum()))
        if cfg["H"] * cfg["W"] < 5000:
            store[f"disp/{name}/depth"] = depth_pred
        print(name, store[f"disp/{name}/scale_shift"], store[f"disp/{name}/metrics"])

for name, cfg in NORMALS_EVAL_CASES.items():
    normals_pred, normals_gt = normals_eval_input(cfg)
    cosine_error = metric.compute_cosine_error(normals_pred[None], normals_gt[None], masked=True)
    store[f"normals/{name}/metrics"] = np.array([float(f(cosine_error)) for f in NORMALS_FUNCS])
    store[f"normals/{name}/n_valid"] = np.array(cosine_error.shape[0])
    if name == PIXEL_CASE:
        store[f"normals/{name}/errors"] = cosine_error
    print(name, cosine_error.shape[0], store[f"normals/{name}/metrics"])

for name, cfg in IID_EVAL_CASES.items():
    target_pred, target_gt, valid_mask = iid_eval_input(cfg)
    t = cfg.get("transform")
    if t == "srgb2linear":                                  # script/iid/eval.py:183-196 (image_util.py:144-149)
        target_gt, target_pred = target_gt ** 2.2, target_pred ** 2.2
    elif t == "linear2srgb":
        target_gt, target_pred = target_gt ** (1.0 / 2.2), target_pred ** (1.0 / 2.2)
    value = metric.compute_iid_metric(target_pred.clone(), target_gt.clone(), cfg["target"], "psnr", psnr, valid_mask)
    store[f"iid/{name}/psnr"] = np.array(value)
    if cfg["target"] in ("shading", "residual"):
        store[f"iid/{name}/lstsq_scale"] = np.array(
            metric.compute_alignment_scale(target_pred, target_gt, valid_mask).item())
    print(name, value)

np.savez_compressed(out_dir / "eval_golden.npz", **store)
print("wrote", out_dir / "eval_golden.npz", sum(v.nbytes for v in store.values()) / 1e6, "MB raw")
