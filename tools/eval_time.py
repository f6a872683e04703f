"""Time one sample of each device evaluation path added for normals, IID and disparity-aligned depth against the reference's
path on the same GPU (the torch / numpy restatement in tests/eval_reference.py with CUDA tensors; the normals median is
numpy's on the host, as compute_cosine_error hands the map to np.median). Each timing covers the call from device-resident
inputs to host metrics, host clock around work that ends in a device synchronisation; median of --reps calls after
--warmup. Writes one JSON line per path, with the GPU's name and power limit read in the same process.

    python tools/eval_time.py [--reps 20] [--warmup 3] [--out profiles/r04_eval_time.jsonl]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from marigold_b200.evaluation import evaluate_depth, evaluate_iid, evaluate_normals  # noqa: E402
from tests import eval_reference as R  # noqa: E402
from tests.golden.eval_cases import (DISPARITY_CASES, IID_EVAL_CASES, NORMALS_EVAL_CASES, disparity_input,  # noqa: E402
                                     iid_eval_input, normals_eval_input)


def _time(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3, float(np.min(ts)) * 1e3


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r04_eval_time.jsonl"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/eval_time.py needs a CUDA device")
    gpu = _gpu()
    rows = []

    pred, gt = normals_eval_input(NORMALS_EVAL_CASES["n480x640"])
    pred, gt = pred.cuda(), gt.cuda()
    rows.append(("normals 480x640", lambda: evaluate_normals(pred, gt),
                 lambda: R.normals_metrics(R.cosine_error(pred, gt))))

    iid = {t: iid_eval_input(IID_EVAL_CASES[f"{t}_768x1024"]) for t in ("albedo", "shading", "residual")}
    iid = {t: (p.cuda(), g.cuda(), None if m is None else m.cuda()) for t, (p, g, m) in iid.items()}
    tr = {t: IID_EVAL_CASES[f"{t}_768x1024"].get("transform") for t in iid}
    rows.append(("iid 3 targets 768x1024 psnr",
                 lambda: [evaluate_iid(p, g, t, m, tr[t]) for t, (p, g, m) in iid.items()],
                 lambda: [R.eval_iid_psnr(p, g, t, m, tr[t]) for t, (p, g, m) in iid.items()]))

    cfg = DISPARITY_CASES["d480x640"]
    dp, dg, dm = disparity_input(cfg)
    tp, tg, tm = torch.from_numpy(dp).cuda(), torch.from_numpy(dg).cuda(), torch.from_numpy(dm).cuda()
    # the reference loads the prediction from disk as numpy and fits on the host; its metric tensors live on the GPU
    rows.append(("depth least_square_disparity 480x640",
                 lambda: evaluate_depth(tp, tg, tm, alignment="least_square_disparity", min_depth=cfg["dmin"],
                                        max_depth=cfg["dmax"]),
                 lambda: R.eval_depth_disparity(dp, dg, dm, cfg["dmin"], cfg["dmax"], device="cuda")))

    out = Path(a.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    with np.errstate(divide="ignore", invalid="ignore"), open(out, "a") as f:
        for name, ours, ref in rows:
            o_med, o_min = _time(ours, a.reps, a.warmup)
            r_med, r_min = _time(ref, a.reps, a.warmup)
            line = {"path": name, "device_ms_median": round(o_med, 4), "device_ms_min": round(o_min, 4),
                    "reference_ms_median": round(r_med, 4), "reference_ms_min": round(r_min, 4),
                    "speedup_median": round(r_med / o_med, 2), "reps": a.reps, "gpu": gpu}
            print(json.dumps(line))
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
