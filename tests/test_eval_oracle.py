"""The reference restatement of tests/eval_reference.py reproduces what the reference's own evaluation code returned
(tests/golden/eval_golden.npz, written by tests/golden/make_eval_golden.py). Both run the same float32 torch / numpy
operations in the same order on the CPU, so every value must agree bit for bit; NaN (the reference's inf - inf) equals
NaN. torch splits large CPU reductions over its threads, so the tests run with the generator's 4 threads."""
from pathlib import Path

import numpy as np
import pytest
import torch

from tests import eval_reference as R
from tests.golden.eval_cases import (DISPARITY_CASES, IID_EVAL_CASES, NORMALS_EVAL_CASES, PIXEL_CASE, disparity_input,
                                     iid_eval_input, normals_eval_input)

GOLD = np.load(Path(__file__).resolve().parent / "golden" / "eval_golden.npz")


@pytest.fixture(autouse=True)
def _four_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(4)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", list(DISPARITY_CASES))
def test_disparity_depth_eval_matches_golden(name):
    cfg = DISPARITY_CASES[name]
    pred, gt, mask = disparity_input(cfg)
    with np.errstate(divide="ignore", invalid="ignore"):
        metrics, scale, shift, depth = R.eval_depth_disparity(pred, gt, mask, cfg["dmin"], cfg["dmax"])
    np.testing.assert_array_equal(np.array([metrics[k] for k in R.DEPTH_METRICS]), GOLD[f"disp/{name}/metrics"])
    np.testing.assert_array_equal(np.array([scale, shift]), GOLD[f"disp/{name}/scale_shift"])
    if f"disp/{name}/depth" in GOLD:
        np.testing.assert_array_equal(depth, GOLD[f"disp/{name}/depth"])


@pytest.mark.parametrize("name", list(NORMALS_EVAL_CASES))
def test_normals_eval_matches_golden(name):
    pred, gt = normals_eval_input(NORMALS_EVAL_CASES[name])
    err = R.cosine_error(pred, gt)
    assert err.shape[0] == int(GOLD[f"normals/{name}/n_valid"])
    m = R.normals_metrics(err)
    np.testing.assert_array_equal(np.array(list(m.values())), GOLD[f"normals/{name}/metrics"])
    if name == PIXEL_CASE:
        np.testing.assert_array_equal(err, GOLD[f"normals/{name}/errors"])


@pytest.mark.parametrize("name", list(IID_EVAL_CASES))
def test_iid_psnr_matches_golden(name):
    cfg = IID_EVAL_CASES[name]
    pred, gt, mask = iid_eval_input(cfg)
    out = R.eval_iid_psnr(pred, gt, cfg["target"], mask, cfg.get("transform"))
    # torch.linalg.lstsq's float32 LAPACK solve is not run-to-run reproducible on the CPU: between identical calls its
    # scale moved by up to 1.5e-3 relative for a 2.4M x 1 system (PSNR by 1.3e-3 dB), and the PSNR of a 5k x 1 system by
    # 1.9e-6 dB. Aligned targets are bounded accordingly; everything else is exact.
    aligned = cfg["target"] in ("shading", "residual")
    big = cfg["H"] * cfg["W"] > 100_000
    tol_psnr, tol_scale = ((5e-3, 5e-3) if big else (1e-4, 1e-5)) if aligned else (0.0, 0.0)
    assert abs(out["psnr"] - float(GOLD[f"iid/{name}/psnr"])) <= tol_psnr or out["psnr"] == float(GOLD[f"iid/{name}/psnr"])
    if cfg["target"] in ("shading", "residual"):
        s = float(GOLD[f"iid/{name}/lstsq_scale"])
        assert abs(out["lstsq_scale"] - s) <= tol_scale * abs(s)
        assert (out["quantile_scale"] == 0) == bool(cfg.get("dark"))


def test_quantile_rank_is_formed_in_float32():
    """torch.quantile's linear interpolation, restated the way the device computes it: rank = f32(0.9) * f32(n - 1),
    floor / ceil, and one fma on either side of weight 0.5 (torch's lerp)."""
    rng = np.random.default_rng(5)
    for n in (1, 2, 7, 1961, 307200, 786432, 1000001):
        x = np.sort(rng.uniform(0, 1, n).astype(np.float32) * np.float32(rng.uniform(0.1, 10)))
        r = np.float32(0.9) * np.float32(n - 1)
        k = int(r)
        w = np.float32(r - np.float32(k))
        a, b = np.float64(x[k]), np.float64(x[min(k + 1, n - 1)])
        d = np.float64(np.float32(b - a))
        q = np.float32(w * d + a) if w < 0.5 else np.float32(b - d * np.float64(np.float32(1 - w)))
        assert q == torch.quantile(torch.from_numpy(x), 0.9).item(), n
