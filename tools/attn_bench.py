"""Self-attention alone (ops.flash_attn64 incl. the split-KV combine pass) at every UNet shape, timed by CUDA-graph
replay of 20 launches as bench.py times its dominant kernels. For each shape: microseconds per call, TF/s, and the
ratio of the tensor floor (4 T^2 64 FLOP per (image, head) at the burst peak) and of the MUFU floor (one exponential
per score at 16 per SM and clock) to the measured time. The GPU name, power limit and SM clock are read in the same
run.

    python tools/attn_bench.py [--arm LABEL] [--rounds N] [--out FILE.jsonl]

To compare two builds, run the script alternately from each build's tree with the same --out.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

# (label, NB, T, C): the four self-attention levels of one member at 768^2, then the batched c3 (8 members) and
# c4 (10 members) grids of the 96^2 level
SHAPES = [
    ("96^2", 1, 9216, 320),
    ("48^2", 1, 2304, 640),
    ("24^2", 1, 576, 1280),
    ("12^2", 1, 144, 1280),
    ("96^2 NB=8", 8, 9216, 320),
    ("96^2 NB=10", 10, 9216, 320),
]
BURST_TFLOPS = 1590.0   # bf16 burst figure bench.py uses without MEASURED_PEAKS.json
MUFU_PER_SM_CLK = 16
SMS = 148


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, sm, smax = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit_w": float(pl), "sm_clock_mhz": float(sm), "sm_clock_max_mhz": float(smax)}
    except Exception as e:  # noqa: BLE001
        return {"gpu_info_error": repr(e)[:200]}


def graph_time_us(torch, launch, n=20, reps=5):
    launch()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        launch()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=s):
            for _ in range(n):
                launch()
    torch.cuda.synchronize()
    gr.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        gr.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (n * reps)


def rel_err(torch, out, qkv, NB, T, C):
    import torch.nn.functional as F
    h = C // 64
    q, k, v = [t.float().reshape(NB, T, h, 64).permute(0, 2, 1, 3) for t in qkv.split(C, dim=1)]
    ref = F.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(NB * T, C)
    return float((out.float() - ref).abs().max() / ref.abs().max())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arm", default="this build", help="label written with every record")
    ap.add_argument("--rounds", type=int, default=1, help="timing passes over all shapes (the first also checks errors)")
    ap.add_argument("--out", default="attn_bench.jsonl")
    a = ap.parse_args()

    import torch
    from marigold_b200 import ops

    info = gpu_info()
    clock_hz = info.get("sm_clock_max_mhz", 1965.0) * 1e6   # the MUFU floor at the boost clock
    print(json.dumps(info), flush=True)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    fout = open(a.out, "a")
    fout.write(json.dumps(info) + "\n")
    g = torch.Generator(device="cuda").manual_seed(0)
    inputs = {s: torch.randn(s[1] * s[2], 3 * s[3], device="cuda", generator=g).to(torch.bfloat16) for s in SHAPES}

    def run(arm, shapes, check):
        for s in shapes:
            label, NB, T, C = s
            qkv = inputs[s]
            us = graph_time_us(torch, lambda: ops.flash_attn64(qkv, NB, T, C, 0.125))
            flop = 4.0 * NB * (C // 64) * T * T * 64
            exps = NB * (C // 64) * T * T
            rec = {"arm": arm, "shape": label, "NB": NB, "T": T, "C": C, "us": round(us, 2),
                   "tflops": round(flop / us / 1e6, 1),
                   "tensor_floor_frac": round(flop / (BURST_TFLOPS * 1e12) / (us * 1e-6), 3),
                   "mufu_floor_frac": round(exps / (MUFU_PER_SM_CLK * SMS * clock_hz) / (us * 1e-6), 3)}
            if check:
                rec["rel_err"] = rel_err(torch, ops.flash_attn64(qkv, NB, T, C, 0.125), qkv, NB, T, C)
            print(json.dumps(rec), flush=True)
            fout.write(json.dumps(rec) + "\n")

    for r in range(a.rounds):
        run(a.arm, SHAPES, check=r == 0)
    print(json.dumps(gpu_info()), flush=True)


if __name__ == "__main__":
    main()
