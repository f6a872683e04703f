"""Benchmark of the Marigold denoising hot path (BASELINE.json metric: denoise-steps/sec @768 px).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config c2|c3|c4|c5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR (--impl b200) writes, after the timed work, what it computed as DIR/<name>.npy (float32): `latent`,
the denoised latents of all members after the last timed step [E, 4, h, w], and the last end-to-end call's prediction
(`depth` or `normals`) with, for E > 1, its `uncertainty`. Weights, image and noise are seeded, so two builds run with the
same arguments can be compared output for output.

--config selects the BASELINE.json configuration (default c2 = configs[1], the headline; the others are the
LCM / normals / 1024-px cases of configs[2..4], same metric, members sharded round-robin over the ranks).

A "step" is one denoising iteration (cat -> UNet -> scheduler.step, reference
marigold/marigold_depth_pipeline.py:456-468) of ONE ensemble member at 768x768 (latent 96x96), the
configuration BASELINE.json quotes the metric on (configs[1]: marigold-depth-v1-1, 768x768, E=1, 50 DDIM
steps, bf16 operands, 1 GPU). With N GPUs every rank runs one member (weak scaling, no collective in the
loop; SURVEY.md §8e) and `value` = N * K / max-over-ranks device time.

Weights are random-init tensors of the SD-2 UNet / SD VAE architecture (no checkpoints offline) and the
image / noise are synthetic: "data": "synthetic". Inputs exceed L2: every step streams the 1.73 GB bf16
UNet weights from HBM (L2 is 126 MB), so no explicit flush is needed between iterations.

One JSON line is printed by rank 0; see DESIGN.md §Measurement for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

F_UNET = {384: 0.418e12, 768: 2.138e12, 1024: 4.658e12}    # algorithmic FLOP per member-step (SURVEY.md App. B)
METRIC = "denoise-steps/sec @768px (UNet forward + scheduler step per ensemble member)"
# BASELINE.json configs[1..4]. ensemble: None = one member per GPU (weak scaling, the headline); a number = that many
# members sharded round-robin over the ranks (rank r takes r, r+G, ...: uneven 2/1 splits for E=10 on 8 GPUs).
CONFIGS = {
    "c2": dict(name="marigold-depth-v1-1, 768x768, ensemble_size=1 member per GPU, 50-step DDIM (trailing, zero-SNR, v-pred)",
               res=768, sched="ddim", sched_steps=50, ensemble=None, task="depth", images=1),
    "c3": dict(name="marigold-depth-lcm-v1-0, 768x768, ensemble_size=8, 4-step LCM", res=768, sched="lcm", sched_steps=4,
               ensemble=8, task="depth", images=1),
    "c4": dict(name="marigold-normals-v1-1, 768x768, ensemble_size=10, 10-step DDIM", res=768, sched="ddim",
               sched_steps=10, ensemble=10, task="normals", images=1),
    "c5": dict(name="marigold-depth-v1-1, 1024x1024, ensemble_size=10, 50-step DDIM, image batch (bounded sample: 2 of 16 "
                    "images end to end)", res=1024, sched="ddim", sched_steps=50, ensemble=10, task="depth", images=2),
}
RES, SCHEDULE_STEPS = 768, 50           # headline values; run_b200 / run_reference use the selected config


def usable_cores() -> int:
    """Cores this process may actually use (affinity mask and cgroup CPU quota), not os.cpu_count()."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:  # noqa: BLE001
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:  # noqa: BLE001
        pass
    return max(1, n)


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:  # noqa: BLE001
        pass
    return "unknown"


def synthetic_image(S: int, seed: int = 1234):
    """uint8 [1,3,S,S]: smooth sinusoids + rectangles + pixel noise (SURVEY.md 8(d))."""
    import numpy as np
    import torch

    rng = np.random.default_rng(seed)
    yy, xx = np.meshgrid(np.linspace(0, 1, S), np.linspace(0, 1, S), indexing="ij")
    img = np.zeros((3, S, S))
    for _ in range(6):
        fx, fy, ph = rng.uniform(0.5, 4, 2).tolist() + [rng.uniform(0, 6.28)]
        amp = rng.uniform(20, 50, 3)
        img += amp[:, None, None] * np.sin(2 * np.pi * (fx * xx + fy * yy) + ph)[None]
    img += 128
    for _ in range(5):
        x0, y0 = rng.integers(0, S - 8, 2)
        w, h = rng.integers(8, max(9, S // 3), 2)
        img[:, y0:y0 + h, x0:x0 + w] = rng.uniform(0, 255, 3)[:, None, None]
    img += rng.normal(0, 4, img.shape)
    return torch.from_numpy(np.clip(img, 0, 255).astype(np.uint8))[None]


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"tflops_sustained": d.get("bf16_tflops_sustained"), "tflops_burst": d.get("bf16_tflops"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:  # noqa: BLE001
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


DUMP_LIMIT_BYTES = 64 << 20


def _dump_outputs(out_dir, arrays):
    """Save each array of `arrays` (name -> tensor or ndarray; None entries skipped) as out_dir/<name>.npy in float32."""
    import numpy as np

    arrs = {}
    for name, a in arrays.items():
        if a is not None:
            a = a.detach().cpu().numpy() if hasattr(a, "detach") else a
            arrs[name] = np.ascontiguousarray(a, dtype=np.float32)
    total = sum(a.nbytes for a in arrs.values())
    assert total <= DUMP_LIMIT_BYTES, f"outputs of {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte dump limit"
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrs.items():
        np.save(d / f"{name}.npy", a)


def _build_models(kind="full"):
    """Random-init weights of the real architecture (torch default init, seed 0): the oracle modules are only the
    weight generator here (and the checker of the cpu_baseline / --impl reference legs)."""
    import torch

    from oracle.unet import UNet2DConditionOracle, UNetConfig
    from oracle.vae import AutoencoderKLOracle, VAEConfig

    torch.manual_seed(0)
    unet = UNet2DConditionOracle(UNetConfig()).eval()
    vae = AutoencoderKLOracle(VAEConfig()).eval()
    text = torch.randn(1, 2, 1024, generator=torch.Generator().manual_seed(7))
    return unet, vae, text


def _engine(unet, vae, text):
    from marigold_b200.engine import Engine, EngineConfig

    eng = Engine(EngineConfig())
    eng.load_state_dict("unet", unet.state_dict())
    eng.load_state_dict("vae", vae.state_dict())
    eng.finalize()
    eng.set_text_embedding(text)
    return eng


def _scheduler(cfg):
    from marigold_b200.schedulers import DDIMScheduler, LCMScheduler

    return LCMScheduler() if cfg["sched"] == "lcm" else DDIMScheduler()


def _tables(cfg, total):
    """Coefficient tables of the configuration's schedule, cycled to `total` entries."""
    import numpy as np

    s = _scheduler(cfg)
    s.set_timesteps(cfg["sched_steps"])
    kx, kv, kz = s.coefficients()
    idx = np.arange(total) % cfg["sched_steps"]
    return s.timesteps[idx], kx[idx], kv[idx], kz[idx]


# -------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    from marigold_b200 import _lib, parallel
    from marigold_b200.pipeline import MarigoldDepthPipeline, MarigoldNormalsPipeline

    cfg = CONFIGS[args.config]
    res, n_sched = cfg["res"], cfg["sched_steps"]
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    lib = _lib.load()

    torch.set_num_threads(max(1, usable_cores() // max(1, world)))   # N ranks share the box's usable cores
    unet, vae, text = _build_models("full")
    eng = _engine(unet, vae, text)
    del vae                                   # weights live on the device now; only rank 0 keeps the fp32 UNet
    if rank != 0 or (args.no_cpu_baseline and args.no_library_baseline):
        unet = None                           # (the checker of the cpu_baseline / library-baseline legs)
    import gc

    gc.collect()
    K, W = args.steps, args.warmup
    ts, kx, kv, kz = _tables(cfg, W + K)
    eng.set_schedule(ts, kx, kv, kz)

    E = cfg["ensemble"] if cfg["ensemble"] is not None else world            # c2: one member per GPU
    mine = parallel.member_indices(E, rank, world)
    B = len(mine)
    lh = lw = res // 8
    g = torch.Generator().manual_seed(2024)
    noise_all = torch.randn(E, 4, lh, lw, generator=g)                        # member k uses row k on any rank
    step_noise_all = torch.randn(W + K, E, 4, lh, lw, generator=g) if cfg["sched"] == "lcm" else None
    img = synthetic_image(res)
    rgb = (img.float() / 255.0 * 2 - 1).to(dev)
    rgb_latent = eng.encode(rgb).expand(max(B, 1), -1, -1, -1).contiguous()
    target = noise_all[mine].to(dev).contiguous() if B else None
    sn = step_noise_all[:, mine].to(dev).contiguous() if (step_noise_all is not None and B) else None

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-timed K steps, inputs resident in HBM -------------------------------------------
    if B:
        eng.denoise_range_(rgb_latent, target, 0, W, sn)
    sync_all()
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = lib.mgb_launch_count()
    t_cpu0 = time.perf_counter()
    e0.record()
    if B:
        eng.denoise_range_(rgb_latent, target, W, K, sn)
    e1.record()
    t_enqueue = time.perf_counter() - t_cpu0
    sync_all()
    launches = int(lib.mgb_launch_count() - l0)
    clocks = sampler.stop()
    ms_local = e0.elapsed_time(e1)
    ms = parallel.barrier_max_ms(ms_local, dev)
    if B:
        assert torch.isfinite(target).all(), "non-finite latent after the timed region"
    latent = None
    if args.dump_outputs:                            # a collective when world > 1: every rank takes part
        local = target if B else torch.empty(0, 4, lh, lw, device=dev)
        latent = parallel.gather_members(local, E).cpu()
    value = E * K / (ms / 1e3)                       # member-steps of ALL ranks / max-over-ranks device time

    # ---- end to end through the public pipeline API: host image in, numpy map out --------------
    n_e2e = n_sched                                   # the whole call the config names (c2: 50 DDIM steps)
    sched = _scheduler(cfg)
    Pipe = MarigoldNormalsPipeline if cfg["task"] == "normals" else MarigoldDepthPipeline
    pipe = Pipe(eng, sched, text, default_denoising_steps=n_e2e, default_processing_resolution=res)
    img_pinned = img.pin_memory()
    noise_pinned = noise_all.pin_memory()
    kw = dict(ensemble_size=E, noise=noise_pinned, show_progress_bar=False)
    if cfg["task"] == "depth":
        kw["color_map"] = None
    if cfg["sched"] == "lcm" and n_e2e > 1:
        kw["step_noise"] = step_noise_all[: n_e2e - 1].pin_memory()
    import logging

    logging.disable(logging.WARNING)
    pipe(img_pinned, **kw)                                                   # warm-up
    sync_all()
    reps = max(2, cfg["images"])
    t0 = time.perf_counter()
    for _ in range(reps):
        out = pipe(img_pinned, **kw)
    torch.cuda.synchronize()
    t_e2e_local = (time.perf_counter() - t0) / reps
    t_e2e = parallel.barrier_max_ms(t_e2e_local * 1e3, dev) / 1e3
    e2e_value = E * n_e2e / t_e2e
    h2d = img_pinned.numel() * img_pinned.element_size() + len(mine) * 4 * lh * lw * 4
    res_np = out.normals_np if cfg["task"] == "normals" else out.depth_np
    d2h = res_np.size * 4
    if rank == 0 and args.dump_outputs:
        _dump_outputs(args.dump_outputs, {"latent": latent, cfg["task"]: res_np, "uncertainty": out.uncertainty})

    # ---- dominant kernels alone (CUDA-graph replay => pure device time) ---------------------------
    kern = None
    if rank == 0 and not args.no_kernel_roofline:
        kern = _dominant_kernel_roofline(torch)

    # ---- the same graph through torch's library kernels (cuDNN / cuBLAS / SDPA, bf16) on this GPU ----
    libbase = None
    if rank == 0 and not args.no_library_baseline:
        libbase = _library_baseline(unet, text, res, min(K, 10))

    # ---- CPU baseline (oracle port) on a bounded sample ------------------------------------------
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = _cpu_baseline(unet, text, steps=1, res=res)
    eng.close()

    if rank == 0:
        pk = _peaks()
        achieved = E * K * F_UNET[res] / (ms / 1e3) / 1e12
        peak = pk["tflops_sustained"] * world
        line = {
            "metric": METRIC, "value": value, "unit": "denoise-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak" if cfg["ensemble"] is None else "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": cfg["name"] + " — SD-2 UNet 865.9M + SD VAE architecture", "id": args.config,
                       "members_total": E, "members_this_rank": B, "latent": [lh, lw],
                       "parallelism": f"members-dp{world}",
                       "l2": "inputs > L2: 1.73 GB of bf16 weights stream from HBM every step",
                       "weights": "random init (torch default init, seed 0)"},
            "clocks": clocks,
            "gpu_launches": launches,
            "cpu_enqueue_ms_per_step": t_enqueue * 1e3 / K,
            "e2e": {"value": e2e_value, "unit": "denoise-steps/s", "h2d_bytes_per_step": h2d / n_e2e,
                    "d2h_bytes_per_step": d2h / n_e2e, "seconds_per_image": t_e2e, "steps_per_call": n_e2e,
                    "images_timed": reps,
                    "includes": "H2D image+noise, resize/normalise, VAE encode, denoise loop, VAE decode, "
                                + ("all-gather, " if world > 1 else "") + ("ensemble, " if E > 1 else "")
                                + "resize, D2H result"},
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": None,
                         "what": f"whole fused UNet step (all kernels), algorithmic FLOP {F_UNET[res]:.4g} per member-step",
                         "peak_source": pk["source"] + ", bf16_tflops_sustained x n_gpus",
                         "dominant_kernel": kern[0] if kern else None,
                         "kernels": kern},
            "gpu_library_baseline": libbase,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _graph_time_us(torch, launch, n=20, reps=5):
    """Average device time of `launch` from a CUDA graph of n launches (no host gaps)."""
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


def _library_baseline(unet, text, res, steps):
    """Informational GPU yardstick (SURVEY.md 2.3 / 8d): the oracle graph of one UNet + DDIM step run by torch in bf16 on
    the same B200 — cuDNN convolutions, cuBLAS linears, SDPA attention, eager launches — i.e. what the reference pipeline
    executes with torch_dtype=bfloat16. Not part of the product path."""
    import copy

    import torch

    from oracle.schedulers import DDIMSchedulerOracle

    if unet is None:
        return None
    try:
        m = copy.deepcopy(unet).to("cuda", torch.bfloat16)
        ctx = text.to("cuda", torch.bfloat16)
        lh = res // 8
        g = torch.Generator().manual_seed(1)
        x = torch.randn(1, 4, lh, lh, generator=g).to("cuda", torch.bfloat16)
        rgb = torch.randn(1, 4, lh, lh, generator=g).to("cuda", torch.bfloat16)
        o = DDIMSchedulerOracle()
        o.set_timesteps(50)
        with torch.no_grad():
            for i in range(3):
                t = o.timesteps[i]
                x = o.step(m(torch.cat([rgb, x], 1), t, ctx), t, x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                t = o.timesteps[3 + i]
                x = o.step(m(torch.cat([rgb, x], 1), t, ctx), t, x)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        del m
        torch.cuda.empty_cache()
        return {"value": 1e3 / ms, "unit": "denoise-steps/s", "ms_per_step": ms, "steps": steps,
                "what": f"oracle UNet + DDIM graph, torch {torch.__version__} bf16 (cuDNN / cuBLAS / SDPA), eager, 1 member, "
                        f"{res}x{res}, same GPU"}
    except Exception as e:  # noqa: BLE001
        return {"unavailable": repr(e)[:200]}


def _dominant_kernel_roofline(torch):
    """The two kernels that dominate a 768-px UNet step BY TIME, each timed alone from a CUDA graph of 20 launches
    against the burst peak: (1) flash self-attention over the 9216 latent tokens (5 launches x ~0.2 ms per step),
    (2) the top-level 3x3 conv 320 -> 320 @ 96x96 (16 launches per step)."""
    from marigold_b200 import _lib, ops
    from marigold_b200._lib import check, ptr, stream_ptr

    pk = _peaks()
    lib = _lib.load()
    out = []
    # (1) attention: qkv [9216, 960] bf16, 5 heads of 64; algorithmic FLOP 4 T^2 C
    T, C = 9216, 320
    qkv = torch.randn(T, 3 * C, device="cuda").to(torch.bfloat16)
    us = _graph_time_us(torch, lambda: ops.flash_attn64(qkv, 1, T, C, 0.125))
    flop = 4.0 * T * T * C
    ach = flop / (us * 1e-6) / 1e12
    out.append({"kernel": "flash_attn64_kernel + attn_combine_kernel (self-attention, T=9216, 5 heads x 64)",
                "us_per_launch": us, "achieved": ach, "peak": pk["tflops_burst"], "unit": "TFLOP/s",
                "frac": ach / pk["tflops_burst"], "share_of_step": "5 launches/step",
                "peak_source": pk["source"] + ", bf16_tflops (burst: kernel timed alone)",
                "traffic": None, "traffic_source": "profiles/r02_kernel_table.md (ncu --set full, dram read+write)"})
    # (2) conv
    NB, H, W_, Cc = 1, 96, 96, 320
    x = torch.randn(NB, H, W_, Cc, device="cuda").to(torch.bfloat16)
    w = ops.pack_conv_weight((torch.randn(Cc, Cc, 3, 3, device="cuda") / (9 * Cc) ** 0.5).to(torch.bfloat16))
    b = torch.randn(Cc, device="cuda")
    o = torch.empty(NB, H, W_, Cc, dtype=torch.float32, device="cuda")

    def launch():
        check(lib.mgb_op_conv2d(ptr(x), ptr(w), ptr(b), None, ptr(o), None, NB, H, W_, Cc, Cc, 0, 0, 0, 0, 0, None,
                                stream_ptr()), "mgb_op_conv2d")

    us = _graph_time_us(torch, launch)
    flop = 2.0 * NB * H * W_ * Cc * Cc * 9
    ach = flop / (us * 1e-6) / 1e12
    out.append({"kernel": "gemm_tc_kernel<160> (implicit-GEMM conv3x3 320->320 @96x96)", "us_per_launch": us,
                "achieved": ach, "peak": pk["tflops_burst"], "unit": "TFLOP/s", "frac": ach / pk["tflops_burst"],
                "share_of_step": "16 launches/step",
                "peak_source": pk["source"] + ", bf16_tflops (burst: kernel timed alone)",
                # one `ncu --set full` capture of this launch: dram__bytes_read.sum + dram__bytes_write.sum. Algorithmic
                # bytes are 19.5e6 (A 5.9e6 bf16, weights 1.8e6, fp32 output 11.8e6): operands and output stay in the
                # 126 MB L2 between kernels, so DRAM sees less than the algorithm moves.
                "traffic": 7791872, "traffic_source": "ncu r01f, dram read+write bytes per launch"})
    return out


def _cpu_baseline(unet, text, steps=1, res=RES):
    """Oracle port (fp32 torch on the host cores) on a bounded sample: `steps` UNet+DDIM steps at `res`."""
    import torch

    from oracle.schedulers import DDIMSchedulerOracle

    torch.set_num_threads(usable_cores())
    lh = res // 8
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 4, lh, lh, generator=g)
    rgb = torch.randn(1, 4, lh, lh, generator=g)
    o = DDIMSchedulerOracle()
    o.set_timesteps(SCHEDULE_STEPS)
    with torch.no_grad():
        t0 = time.perf_counter()
        for i in range(steps):
            t = o.timesteps[i]
            x = o.step(unet(torch.cat([rgb, x], 1), t, text), t, x)
        dt = time.perf_counter() - t0
    return {"value": steps / dt, "unit": "denoise-steps/s", "cores": torch.get_num_threads(), "cpu": cpu_model(),
            "kind": "port", "sample": f"{steps} UNet+DDIM step(s), 1 member, {res}x{res}, fp32 torch CPU oracle (oracle/unet.py), "
                      f"{dt:.1f} s"}


# -------------------------------------------------------------------------------------------------
def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path. The reference pipeline cannot
    be imported offline (diffusers absent), so this is the oracle PORT (kind="port") on all host cores."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import torch

    K, W = args.steps, args.warmup
    unet, vae, text = _build_models("full")
    torch.set_num_threads(usable_cores())
    # bounded sample: pick the resolution so that W + K steps fit in ~4 minutes on this host
    cfg = CONFIGS[args.config]
    target = cfg["res"]
    probe = _cpu_baseline(unet, text, steps=1, res=384)
    t384 = 1.0 / probe["value"]
    budget = 240.0
    res = target if (W + K) * t384 * (F_UNET[target] / F_UNET[384]) < budget else 384
    lh = res // 8
    from oracle.schedulers import DDIMSchedulerOracle

    o = DDIMSchedulerOracle()
    o.set_timesteps(SCHEDULE_STEPS)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 4, lh, lh, generator=g)
    rgb = torch.randn(1, 4, lh, lh, generator=g)
    n_sched = SCHEDULE_STEPS
    with torch.no_grad():
        for i in range(W):
            t = o.timesteps[i % n_sched]
            x = o.step(unet(torch.cat([rgb, x], 1), t, text), t, x)
        t0 = time.perf_counter()
        for i in range(W, W + K):
            t = o.timesteps[i % n_sched]
            x = o.step(unet(torch.cat([rgb, x], 1), t, text), t, x)
        dt = time.perf_counter() - t0
    scale = F_UNET[res] / F_UNET[target]          # FLOP-equivalent steps at the configuration's resolution
    value = K * scale / dt
    sample = (f"{K} UNet+DDIM steps at {res}x{res} (1 member), fp32 torch CPU oracle port; "
              + ("measured at the metric's resolution" if res == target else
                 f"bounded sample: value scaled by F_unet({res})/F_unet({target}) = {scale:.4f} to {target}-px-equivalent "
                 f"steps"))
    cpu = {"value": value, "unit": "denoise-steps/s", "cores": torch.get_num_threads(), "cpu": cpu_model(), "kind": "port",
           "sample": sample}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "denoise-steps/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", args.gpus)), "steps": K, "warmup": W,
            "ms_per_step": dt * 1e3 / K / scale, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["name"] + " — SD-2 UNet 865.9M + SD VAE architecture", "id": args.config,
                       "note": "reference pipeline needs diffusers (absent offline): oracle port on host cores"},
            "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": "denoise-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--no-kernel-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed work, write what it computed as DIR/<name>.npy (float32, <= 64 MB in all)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        # the reference arm picks its resolution from a timing probe, so its outputs are not fixed by the arguments
        ap.error("--dump-outputs needs --impl b200")
    if a.warmup < 3 and a.impl == "b200":
        a.warmup = 3
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
