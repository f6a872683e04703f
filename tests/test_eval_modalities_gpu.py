"""Device evaluation of normals, IID and disparity-aligned depth (`-m gpu`; marigold_b200.evaluation, csrc/eval.cu):
against the goldens the reference's own evaluation code produced (tests/golden/eval_golden.npz), against numpy / torch on
the kernel's own angle map, and the exact order statistic against sorting."""
from pathlib import Path

import numpy as np
import pytest
import torch

from tests import eval_reference as R
from tests.golden.eval_cases import (DISPARITY_CASES, IID_EVAL_CASES, NORMALS_EVAL_CASES, PIXEL_CASE, disparity_input,
                                     iid_eval_input, normals_eval_input)

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).resolve().parent / "golden"
GOLD = np.load(GOLDEN / "eval_golden.npz")

# Tolerances: the deviation measured on a B200 (power limit 1000 W), times a margin.
#  - disparity depth: the fit is double normal equations against the reference's float32 SVD lstsq, and the aligned
#    depth and metrics are double against float32, as in least_square mode. Measured: metrics 5.9e-7 relative, depth map
#    2.4e-7, scale / shift 1e-7.
#  - normals: the device's float32 cosine / acos against torch's CPU kernels. Measured: angles 1.5e-5 deg, cosines
#    2.5e-7; the rounded metrics were identical. A 1-ulp cosine near 0 deg would be ~0.02 deg, hence the angle bound;
#    a rounded metric may still move by one unit of the 4th decimal.
#  - PSNR: double sums of the float32 squared errors against torch's float32 sum; powf against torch's pow. Measured:
#    2.8e-6 dB; the lstsq scale 2.2e-7 relative.
DISP_REL = 5e-6
NORMALS_METRIC_ABS = 1e-4
ANGLE_ABS = 0.025
COS_ABS = 1e-6
PSNR_ABS = 2e-5
PSNR_ABS_BIG = 5e-3
LSTSQ_REL = 2e-6


def _np_median32(x: np.ndarray) -> float:
    return float(np.median(x))


# ---- depth, least_square_disparity ----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(DISPARITY_CASES))
def test_disparity_alignment_matches_golden(name):
    from marigold_b200.evaluation import METRIC_NAMES, evaluate_depth

    cfg = DISPARITY_CASES[name]
    pred, gt, mask = disparity_input(cfg)
    got, info, depth = evaluate_depth(torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda(), torch.from_numpy(mask).cuda(),
                                      alignment="least_square_disparity", min_depth=cfg["dmin"], max_depth=cfg["dmax"],
                                      return_aligned=True)
    assert info["n_valid"] == int(mask.sum())
    scale, shift = GOLD[f"disp/{name}/scale_shift"]
    assert abs(info["scale"] - scale) <= DISP_REL * max(abs(scale), 1e-3), (info, scale)
    assert abs(info["shift"] - shift) <= DISP_REL * max(abs(scale), 1e-3), (info, shift)
    for k, ref in zip(METRIC_NAMES, GOLD[f"disp/{name}/metrics"]):
        if np.isnan(ref):
            continue   # silog's inf - inf with gt == 0 inside the mask: the device clamps the negative variance term to 0
        if np.isinf(ref):
            assert got[k] == ref, (k, got[k])
        else:
            assert abs(got[k] - ref) <= DISP_REL * max(1.0, abs(ref)), (k, got[k], ref)
    if f"disp/{name}/depth" in GOLD:
        ref = GOLD[f"disp/{name}/depth"]
        d = depth.cpu().numpy()
        assert np.all(np.abs(d - ref) <= DISP_REL * np.maximum(1.0, np.abs(ref)))
    if cfg.get("all_negative"):
        assert info["scale"] == 0.0 and info["shift"] == 0.0        # lstsq of an empty system
        assert np.all(depth.cpu().numpy() == np.float32(cfg["dmax"]))


# ---- normals --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(NORMALS_EVAL_CASES))
def test_normals_metrics_match_golden(name):
    from marigold_b200.evaluation import NORMALS_METRIC_NAMES, evaluate_normals

    pred, gt = normals_eval_input(NORMALS_EVAL_CASES[name])
    got, info, ang = evaluate_normals(pred[None].cuda(), gt.cuda(), return_errors=True)
    assert info["n_valid"] == int(GOLD[f"normals/{name}/n_valid"])
    for k, ref in zip(NORMALS_METRIC_NAMES, GOLD[f"normals/{name}/metrics"]):
        assert abs(got[k] - ref) <= NORMALS_METRIC_ABS, (k, got[k], ref)
    a = ang.cpu().numpy()
    valid = (gt.norm(dim=0) > 0).numpy()
    assert np.array_equal(~np.isnan(a), valid)
    if name == PIXEL_CASE:
        np.testing.assert_allclose(a[valid], GOLD[f"normals/{name}/errors"], rtol=0, atol=ANGLE_ABS)


@pytest.mark.parametrize("name", list(NORMALS_EVAL_CASES))
def test_normals_metrics_match_numpy_on_the_kernels_angles(name):
    """Median, threshold percentages and n_valid equal numpy's on angles_out exactly; mean and rmse within 1e-4."""
    from marigold_b200.evaluation import normals_raw

    pred, gt = normals_eval_input(NORMALS_EVAL_CASES[name])
    out, ang = normals_raw(pred.cuda(), gt.cuda(), True)
    a = ang.cpu().numpy().reshape(-1)
    e = a[~np.isnan(a)]
    assert out[0] == e.shape[0]
    assert out[2] == _np_median32(e)
    for i, t in enumerate((5, 7.5, 11.25, 22.5, 30)):
        assert out[4 + i] == 100.0 * (np.sum(e < t) / e.shape[0])
    assert abs(out[1] - float(np.average(e))) <= 1e-4
    assert abs(out[3] - float(np.sqrt(np.sum(e * e) / e.shape[0]))) <= 1e-4


def test_angle_map_against_reference_cosine_error():
    """Per pixel against compute_cosine_error's torch ops on the CPU: the cosine agrees to a few float32 ulps, which near 0
    deg the arccos turns into up to ~0.02 deg."""
    pred, gt = normals_eval_input(NORMALS_EVAL_CASES["n480x640"])
    from marigold_b200.evaluation import normals_raw

    _, ang = normals_raw(pred.cuda(), gt.cuda(), True)
    a = ang.cpu().numpy().reshape(-1)
    ref = R.cosine_error(pred, gt)
    got = a[~np.isnan(a)]
    cg, cr = np.cos(np.deg2rad(got.astype(np.float64))), np.cos(np.deg2rad(ref.astype(np.float64)))
    assert np.abs(cg - cr).max() <= COS_ABS
    assert np.abs(got - ref).max() <= ANGLE_ABS


# ---- order statistic: median through the normals path ---------------------------------------------------------------
def _angles_case(kind: str):
    g = torch.Generator().manual_seed(11)
    H, W = 96, 160
    gt = torch.zeros(3, H, W)
    gt[2] = 1.0
    pred = gt.clone()
    if kind == "all_equal":
        pred[0] = 0.3
    elif kind == "ties_on_boundary":                       # three angles; the middle ranks straddle a run boundary
        n = H * W
        v = torch.zeros(n)
        v[: n // 2] = 0.2
        v[n // 2:] = 0.5
        v[n // 2 + 100: n // 2 + 200] = 0.9
        pred[0] = v[torch.randperm(n, generator=g)].reshape(H, W)
    elif kind == "ties_inside_run":
        n = H * W
        v = torch.full((n,), 0.4)
        v[: n // 3] = 0.1
        v[-n // 3:] = 0.7
        pred[0] = v[torch.randperm(n, generator=g)].reshape(H, W)
    elif kind == "one_valid":
        gt[:] = 0
        gt[:, 5, 7] = torch.tensor([0.1, 0.2, 0.9])
        pred[0] = 0.25
    elif kind == "odd_count":
        gt[:, 0, 0] = 0
        pred[0] = torch.rand(H, W, generator=g)
    return pred, gt


@pytest.mark.parametrize("kind", ["all_equal", "ties_on_boundary", "ties_inside_run", "one_valid", "odd_count"])
def test_median_equals_sort(kind):
    from marigold_b200.evaluation import normals_raw

    pred, gt = _angles_case(kind)
    out, ang = normals_raw(pred.cuda(), gt.cuda(), True)
    a = ang.cpu().reshape(-1)
    e = torch.sort(a[~torch.isnan(a)]).values.numpy()
    n = e.shape[0]
    ref = e[(n - 1) // 2] if n % 2 else (np.float32(e[n // 2 - 1] + e[n // 2]) / np.float32(2))
    assert out[2] == float(ref) == _np_median32(e)


def test_normals_without_valid_pixels_is_nan():
    from marigold_b200.evaluation import evaluate_normals

    got, info = evaluate_normals(torch.ones(3, 8, 8).cuda(), torch.zeros(3, 8, 8).cuda())
    assert info["n_valid"] == 0 and all(np.isnan(v) for v in got.values())


# ---- order statistic: quantile through the IID path -----------------------------------------------------------------
def _sorted_quantile(b: torch.Tensor) -> float:
    s = torch.sort(b).values.numpy()
    n = s.shape[0]
    r = np.float32(0.9) * np.float32(n - 1)
    k = int(r)
    w = np.float32(r - np.float32(k))
    a, c = np.float64(s[k]), np.float64(s[min(k + 1, n - 1)])
    d = np.float64(np.float32(c - a))
    return float(np.float32(w * d + a) if w < 0.5 else np.float32(c - d * np.float64(np.float32(1 - w))))


@pytest.mark.parametrize("kind", ["golden_768x1024", "exponent_range", "all_equal", "ties", "one_pixel", "two_pixels"])
def test_quantile_equals_torch_quantile_and_sort(kind):
    from marigold_b200.evaluation import evaluate_iid

    g = torch.Generator().manual_seed(13)
    mask = None
    if kind == "golden_768x1024":
        pred, gt, mask = iid_eval_input(IID_EVAL_CASES["shading_768x1024"])
    else:
        H, W = (5, 7) if kind in ("one_pixel", "two_pixels") else (211, 307)
        if kind == "exponent_range":                        # every binade from subnormals to 1e38, and zeros
            x = torch.pow(10.0, torch.rand(H, W, generator=g, dtype=torch.float64) * 83 - 45).float()
            x[torch.rand(H, W, generator=g) < 0.05] = 0.0
        elif kind == "all_equal":
            x = torch.full((H, W), 0.37)
        elif kind == "ties":
            x = torch.randint(0, 4, (H, W), generator=g).float() / 4
        else:
            x = torch.rand(H, W, generator=g)
        gt = x[None].expand(3, H, W).contiguous()[None]
        pred = gt * 0.5
        if kind in ("one_pixel", "two_pixels"):              # one or two pixels in the mask
            mask = torch.zeros(1, 3, H, W, dtype=torch.bool)
            mask[..., 2, 3] = True
            if kind == "two_pixels":
                mask[..., 4, 0] = True
    _, info = evaluate_iid(pred.cuda(), gt.cuda(), "shading", None if mask is None else mask.cuda())
    b = R.brightness(gt, mask)
    assert info["quantile"] == _sorted_quantile(b) == torch.quantile(b, 0.9).item()


# ---- IID ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(IID_EVAL_CASES))
def test_iid_psnr_matches_golden(name):
    from marigold_b200.evaluation import evaluate_iid

    cfg = IID_EVAL_CASES[name]
    pred, gt, mask = iid_eval_input(cfg)
    got, info = evaluate_iid(pred.cuda(), gt.cuda(), cfg["target"], None if mask is None else mask.cuda(),
                             cfg.get("transform"))
    ref = float(GOLD[f"iid/{name}/psnr"])
    # the reference's float32 CPU lstsq is itself only reproducible to ~1.5e-3 relative at 768 x 1024
    # (tests/test_eval_oracle.py), which moves its PSNR by ~1e-3 dB
    big = cfg["H"] * cfg["W"] > 100_000 and cfg["target"] in ("shading", "residual")
    tol = PSNR_ABS_BIG if big else PSNR_ABS
    assert got["psnr"] == ref if np.isinf(ref) else abs(got["psnr"] - ref) <= tol, (got, ref)
    assert info["n"] == (int(mask.sum()) if mask is not None else pred.numel())
    if cfg["target"] in ("shading", "residual"):
        s = float(GOLD[f"iid/{name}/lstsq_scale"])
        assert abs(info["lstsq_scale"] - s) <= (5e-3 if big else LSTSQ_REL) * abs(s), (info, s)
        # against the exact least-squares scale (float64 sums of the same float32 elements), rounded to float32
        tp, tg = pred.double(), gt.double()
        if cfg.get("transform") == "srgb2linear":
            tp, tg = pred.float() ** 2.2, gt.float() ** 2.2
            tp, tg = tp.double(), tg.double()
        sel = mask if mask is not None else torch.ones_like(pred, dtype=torch.bool)
        exact = float(np.float32((tp[sel] * tg[sel]).sum() / (tp[sel] * tp[sel]).sum()))
        assert abs(info["lstsq_scale"] - exact) <= 1e-6 * abs(exact), (info, exact)
        assert (info["quantile_scale"] == 0) == bool(cfg.get("dark"))
        o = R.eval_iid_psnr(pred, gt, cfg["target"], mask, cfg.get("transform"))
        if cfg.get("transform") is None:                   # same float32 brightness: the quantile is exact
            assert info["quantile"] == o["quantile"] and info["quantile_scale"] == o["quantile_scale"]
    else:
        assert np.isnan(info["lstsq_scale"]) and np.isnan(info["quantile"])


def test_iid_rejects_unknown_transform_and_cpu_tensors():
    from marigold_b200._lib import MgbError
    from marigold_b200.evaluation import evaluate_iid, evaluate_normals

    x = torch.rand(3, 4, 4)
    with pytest.raises(ValueError):
        evaluate_iid(x.cuda(), x.cuda(), "albedo", color_transform="gamma")
    with pytest.raises(MgbError):
        evaluate_iid(x, x, "albedo")
    with pytest.raises(MgbError):
        evaluate_normals(x, x)


# ---- run-to-run reproducibility -------------------------------------------------------------------------------------
def test_two_calls_give_identical_bits():
    from marigold_b200.evaluation import evaluate_depth, evaluate_iid, normals_raw

    pred, gt = normals_eval_input(NORMALS_EVAL_CASES["n480x640"])
    o1, a1 = normals_raw(pred.cuda(), gt.cuda(), True)
    o2, a2 = normals_raw(pred.cuda(), gt.cuda(), True)
    assert np.array_equal(o1, o2) and torch.equal(a1.isnan(), a2.isnan())
    assert torch.equal(torch.nan_to_num(a1), torch.nan_to_num(a2))
    p, g, m = iid_eval_input(IID_EVAL_CASES["residual_768x1024"])
    r1 = evaluate_iid(p.cuda(), g.cuda(), "residual")
    r2 = evaluate_iid(p.cuda(), g.cuda(), "residual")
    assert r1 == r2
    dp, dg, dm = disparity_input(DISPARITY_CASES["d480x640"])
    args = (torch.from_numpy(dp).cuda(), torch.from_numpy(dg).cuda(), torch.from_numpy(dm).cuda())
    d1 = evaluate_depth(*args, alignment="least_square_disparity", return_aligned=True)
    d2 = evaluate_depth(*args, alignment="least_square_disparity", return_aligned=True)
    assert d1[0] == d2[0] and d1[1] == d2[1] and torch.equal(d1[2], d2[2])


# ---- depth modes 0 / 1 are unchanged --------------------------------------------------------------------------------
def _depth_mode_inputs(align: bool):
    """The inputs of tests/test_image_eval_gpu.py::test_alignment_and_metrics_match_reference_functions."""
    rng = np.random.default_rng(3)
    H, W = 480, 640
    yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
    gt = (1.0 + 4.0 * (0.5 + 0.4 * np.sin(3 * xx + 2 * yy)) + 0.05 * rng.standard_normal((H, W))).astype(np.float32)
    pred = (((gt - 0.7) / 5.1) + 0.02 * rng.standard_normal((H, W))).astype(np.float32)
    if not align:
        pred = (gt * (1 + 0.05 * rng.standard_normal((H, W)))).astype(np.float32)
    mask = rng.uniform(size=(H, W)) > 0.2
    return pred, gt, mask


@pytest.mark.parametrize("align", [True, False])
@pytest.mark.parametrize("with_mask", [True, False])
def test_depth_modes_0_1_bits_unchanged(align, with_mask):
    """mgb_eval_depth with alignment 0 / 1 returns the bits the library returned before disparity mode existed
    (tests/golden/eval_depth_modes.npz: the 13 outputs and a SHA-256 of the aligned map, recorded on a B200)."""
    import hashlib

    from marigold_b200.evaluation import _run

    stored = np.load(GOLDEN / "eval_depth_modes.npz")
    pred, gt, mask = _depth_mode_inputs(align)
    out, aligned = _run(torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda(),
                        torch.from_numpy(mask).cuda() if with_mask else None, int(align), 0.5, 6.0, True)
    key = f"align{int(align)}_mask{int(with_mask)}"
    assert np.array_equal(out.view(np.uint64), stored[f"{key}/out"].view(np.uint64))
    digest = np.frombuffer(hashlib.sha256(aligned.cpu().numpy().tobytes()).digest(), dtype=np.uint8)
    assert np.array_equal(digest, stored[f"{key}/aligned_sha256"])
