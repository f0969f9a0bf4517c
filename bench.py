#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 diffusion backend (BASELINE.json: SDXL-base 1024x1024, 30 Euler-a
steps, batch 8 per GPU, images/sec; UNet ms/step).

    python bench.py --gpus N --steps K --warmup W            # our arm (N>1: launched under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port) on host cores

One bench "step" = one complete txt2img batch: initial latent -> 30 x (UNet forward at batch 16 [uncond|cond] +
fused CFG/Euler-a update) -> VAE decode of 8 images.  Data is synthetic: random-init SDXL UNet/VAE weights of the
reference architecture, N(0,1) latents/noise, N(0,1) conditioning.

Printed JSON (one line, rank 0):
  value      images/sec over all ranks, inputs resident in HBM when the timed region starts
  e2e        the same job through the public API (Txt2ImgPipeline.generate) fed from pinned HOST buffers, with the
             host->device copies and the device->host read of the images inside the timed region
  roofline   the dominant kernel family (tcgen05 GEMM/implicit-GEMM conv): algorithmic FLOPs / CUDA-event time of
             its launches in one instrumented (eager, un-graphed) job step, against the measured dense peak
  cpu_baseline  the oracle port timed on this box's host cores on a bounded sample (N=1, rank 0)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "images_per_sec_sdxl_1024_euler_a_30steps_batch8"
UNIT = "images/s"


def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        peaks.update({k: p[k] for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in p})
        peaks["source"] = "measured"
    except Exception:
        pass
    return peaks


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = []
        reasons = set()
        mx = 0.0
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        busy = [v for v in sm if v > 500] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def usable_cores() -> int:
    """Cores this process may actually use: affinity mask capped by the cgroup CPU quota (os.cpu_count() reports
    the host's cores even inside a CPU-limited container, which would oversubscribe the ATen thread pool)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def cpu_baseline_sample(latent_hw: int, threads: int):
    """Oracle port (the reference's CPU arithmetic: ATen fp32) on a bounded sample: ONE SDXL UNet forward of one
    sample at the benchmark's latent size.  Returns seconds per forward."""
    from oracle import configs as CF
    from oracle import unet as OU
    torch.set_num_threads(threads)
    cfg = CF.SDXL
    sd = OU.random_state_dict(cfg, seed=0)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 4, latent_hw, latent_hw, generator=g)
    ctx = torch.randn(1, 77, cfg["context_dim"], generator=g)
    y = torch.randn(1, cfg["adm_in_channels"], generator=g)
    t = torch.tensor([500.0])

    def fwd():
        with torch.no_grad():
            t0 = time.perf_counter()
            OU.unet_forward(sd, cfg, x, t, ctx, y)
            return time.perf_counter() - t0
    return fwd


def images_per_sec_from_forward(sec_per_sample_forward: float, steps: int = 30) -> float:
    # one image = `steps` sampler steps x 2 UNet sample-forwards (cond + uncond); VAE decode excluded (favours the CPU)
    return 1.0 / (2 * steps * sec_per_sample_forward)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname: str, arrays: dict) -> None:
    """Write each array as DIR/<name>.npy in float32, all of them together within DUMP_LIMIT_BYTES: an array that does not
    fit its share is replaced by a fixed, seeded sample of its flattened elements (the same positions in every run with
    the same arguments, so that two builds can be compared output for output)."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    share = (DUMP_LIMIT_BYTES - 4096 * len(arrays)) // len(arrays) // 4  # elements per array (.npy headers allowed for)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() > share:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(dirname, name + ".npy"), a.numpy())


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = usable_cores()
    fwd = cpu_baseline_sample(128, threads)
    for _ in range(args.warmup if args.warmup is not None else 1):
        fwd()
    k = args.steps if args.steps is not None else 2
    times = [fwd() for _ in range(k)]
    sec = sum(times) / len(times)
    val = images_per_sec_from_forward(sec)
    sample = ("per bench step: 1 SDXL UNet sample-forward (batch 1, latent 128x128, fp32, oracle port = the reference's "
              "ATen CPU path) of the 480 forwards (8 images x 30 steps x cond+uncond) in one batch; images/s = 1/(60*t_fwd)")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": 0, "steps": k,
            "warmup": args.warmup if args.warmup is not None else 1, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "SDXL-base 1024x1024 Euler-a 30 steps batch 8 (CPU sample: one UNet sample-forward)"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def gpu_reference_job(ucfg, vcfg, B, S, hw, cond, uncond, noise, step_noise, sampler, cfg_scale, max_steps=None):
    """Context numbers (not the graded reference arm): the reference's GPU path restated — the oracle port makes the same
    ATen calls Forge makes (F.conv2d -> cuDNN, F.linear -> cuBLAS, F.group_norm, F.scaled_dot_product_attention; fp16 UNet,
    bf16 VAE) and its Denoiser / sample_* loops follow KModel.apply_model + sampling_function_inner + k_diffusion's loop
    with their per-step 0-dim-tensor arithmetic and host syncs.  One COMPLETE job (S sampler steps at UNet batch 2B + VAE
    decode of B images) is timed after a 3-step warm-up; the final latent is returned for the parity check."""
    from oracle import sampling as OS
    from oracle import unet as OU
    from oracle import vae as OV
    from b200forge import synthetic
    dev = noise.device
    sd = synthetic.random_unet_state_dict(ucfg, device=dev, dtype=torch.float16, seed=0)   # same seeds as the timed pipeline
    vsd = synthetic.random_vae_decoder_state_dict(vcfg, device=dev, dtype=torch.bfloat16, seed=1)
    pred = OS.EpsPrediction()
    sig = (OS.get_sigmas_karras(S, float(pred.sigma_min), float(pred.sigma_max)) if sampler == "dpmpp_2m"
           else OS.get_sigmas_uniform(pred, S)).to(dev)
    if max_steps is not None:
        sig = sig[:max_steps + 1]
    c16 = {k: v.to(dev).half() for k, v in cond.items()}
    u16 = {k: v.to(dev).half() for k, v in uncond.items()}

    def unet16(xc, t, c, yy):
        return OU.unet_forward(sd, ucfg, xc, t, c, yy)

    den = OS.Denoiser(unet16, pred, c16, u16, cfg_scale, compute_dtype=torch.float16)
    x0 = noise.to(dev).float() * sig[0]
    it = iter(range(step_noise.shape[0]))
    with torch.no_grad():
        for _ in range(3):
            den(x0, sig[0] * x0.new_ones([B]))
        torch.cuda.synchronize()
        s, m, e = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        s.record()
        if sampler == "dpmpp_2m":
            lat = OS.sample_dpmpp_2m(den, x0.clone(), sig)
        else:
            lat = OS.sample_euler_ancestral(den, x0.clone(), sig, lambda: step_noise[next(it)].to(dev))
        m.record()
        img = torch.cat([OV.decode_first_stage(vsd, vcfg, lat[i:i + 1].bfloat16()) for i in range(B)])
        e.record()
        torch.cuda.synchronize()
    n_steps = sig.numel() - 1
    out = {"unet_ms_per_step": s.elapsed_time(m) / n_steps, "steps_timed": n_steps, "vae_decode_ms": m.elapsed_time(e),
           "job_ms": s.elapsed_time(e), "images_per_s": B / (s.elapsed_time(e) * 1e-3) if n_steps == S else None,
           "what": "oracle port = the reference's ATen/cuDNN/cuBLAS/SDPA calls in fp16 (UNet) / bf16 (VAE), CFG + sampler loop "
                   "with the reference's per-step tensor arithmetic; one complete job after 3 warm-up UNet steps"}
    del sd, vsd, img
    torch.cuda.empty_cache()
    return out, lat


def unet_forward_parity(pipe, ucfg, hw, n, dev):
    """One fused UNet forward at the benchmarked shape [n, 4, hw, hw] against the oracle in fp32 on the same device
    (TF32 off, the engine's own fp16-rounded weights are regenerated from the same seed)."""
    from oracle import unet as OU
    from b200forge import synthetic
    tf = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        g = torch.Generator().manual_seed(123)
        x = torch.randn(n, 4, hw, hw, generator=g).half().to(dev)
        ctx = torch.randn(n, 77, ucfg["context_dim"], generator=g).half().to(dev)
        y = torch.randn(n, ucfg["adm_in_channels"], generator=g).half().to(dev) if ucfg["adm_in_channels"] else None
        t = torch.linspace(999.0, 1.0, n).to(dev)
        out = pipe.unet.forward(x, t, ctx, y).float()
        sd32 = {k: v.float() for k, v in synthetic.random_unet_state_dict(ucfg, device=dev, dtype=torch.float16, seed=0).items()}
        ref = torch.empty_like(out)
        with torch.no_grad():
            for i in range(0, n, 4):
                ref[i:i + 4] = OU.unet_forward(sd32, ucfg, x[i:i + 4].float(), t[i:i + 4], ctx[i:i + 4].float(),
                                               None if y is None else y[i:i + 4].float())
        del sd32
        torch.cuda.empty_cache()
        diff = (out - ref)
        rms = ref.pow(2).mean().sqrt()
        return {"shape": [n, 4, hw, hw], "rel_rms": float(diff.pow(2).mean().sqrt() / rms), "max_abs": float(diff.abs().max()),
                "max_abs_over_ref_rms": float(diff.abs().max() / rms), "finite": bool(torch.isfinite(out).all()),
                "reference": "oracle fp32 on the GPU (TF32 off)"}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf


def attention_vs_sdpa(dev, iters=20):
    """The repo's Dh = 64 attention kernel beside the library the reference calls (F.scaled_dot_product_attention), at the two
    SDXL self-attention shapes, same tensors, CUDA events, L2-sized inputs."""
    from b200forge import ops
    res = {}
    for (b, h, L) in ((16, 10, 4096), (16, 20, 1024)):
        q, k, v = (torch.randn(b, L, h * 64, device=dev, dtype=torch.float16) for _ in range(3))
        qh, kh, vh = (t.view(b, L, h, 64).transpose(1, 2) for t in (q, k, v))
        fl = 4.0 * b * h * L * L * 64

        def timeit(fn):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(iters):
                fn()
            e.record()
            torch.cuda.synchronize()
            return s.elapsed_time(e) / iters

        ours = timeit(lambda: ops.attention(q, k, v, h))
        lib = timeit(lambda: torch.nn.functional.scaled_dot_product_attention(qh, kh, vh))
        res[f"B{b}_H{h}_L{L}_Dh64"] = {"b200_us": ours * 1e3, "b200_tflops": fl / ours / 1e9, "sdpa_us": lib * 1e3,
                                       "sdpa_tflops": fl / lib / 1e9}
    return res


def run_flux(args):
    """BASELINE.json configs[4]: Flux.1-dev (DiT) 1024x1024, 20 Euler steps over the Simple schedule, batch 4 per GPU, bf16,
    distilled guidance 3.5 (CFG 1).  Same contract as the default line; the roofline object is the attention kernel's
    (the config asks for the attention-kernel roofline)."""
    K = args.steps if args.steps is not None else 3
    W = args.warmup if args.warmup is not None else 3
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", torch.cuda.current_device())
    from b200forge import lib, ops, synthetic
    from b200forge.pipeline import FluxTxt2ImgPipeline
    lib.check(lib.load().b200_device_ok())
    peaks = load_peaks()
    B = args.batch if args.batch != 8 else 4
    S = args.sampler_steps if args.sampler_steps != 30 else 20
    hw, Lt = args.size // 8, 256
    cfg = synthetic.FLUX_DEV
    sd = synthetic.random_flux_state_dict(cfg, device=dev)
    vsd = synthetic.random_vae_decoder_state_dict(synthetic.VAE_FLUX, device=dev, dtype=torch.bfloat16, seed=3)
    pipe = FluxTxt2ImgPipeline(cfg, sd, device=dev, vae_cfg=synthetic.VAE_FLUX, vae_state_dict=vsd)
    del sd, vsd
    torch.cuda.empty_cache()
    gens = [torch.Generator().manual_seed(1000 + rank * B + i) for i in range(B)]
    g0 = torch.Generator().manual_seed(7)
    host = {"noise": torch.stack([torch.randn((16, hw, hw), generator=g) for g in gens]).pin_memory(),
            "cond": {"crossattn": torch.randn(B, Lt, cfg["context_in_dim"], generator=g0).bfloat16().pin_memory(),
                     "vector": torch.randn(B, cfg["vec_in_dim"], generator=g0).bfloat16().pin_memory()}}
    devin = {"noise": host["noise"].to(dev), "cond": {k: v.to(dev) for k, v in host["cond"].items()}}
    h2d = host["noise"].numel() * 4 + sum(v.numel() * 2 for v in host["cond"].values())
    out_host = torch.empty((B, args.size, args.size, 3), dtype=torch.float32).pin_memory()
    d2h = out_host.numel() * 4
    gathered = [torch.empty((B, args.size, args.size, 3), dtype=torch.uint8, device=dev) for _ in range(world)] \
        if (dist is not None and rank == 0) else None

    def job(inp):
        return pipe.generate(inp["cond"], inp["noise"], steps=S, guidance=3.5)  # transformer steps + 16-channel VAE decode

    def finish(img):
        if dist is not None:
            from b200forge import dist as bdist
            bdist.gather_images_u8(img, bufs=gathered)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, iters):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(iters):
            fn()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) * 1e-3

    last = {}

    def step_resident():
        last["images"] = job(devin)
        finish(last["images"])

    def step_e2e():
        lat = job(host)
        finish(lat)
        out_host.copy_(lat, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(W):
        step_resident()
    clocks = ClockSampler(torch.cuda.current_device())
    clocks.start()
    l0 = ops.LAUNCHES
    if os.environ.get("B200_PROFILE_TIMED"):  # `ncu --profile-from-start off`: capture exactly the timed region
        torch.cuda.profiler.start()
    sec = timed(step_resident, K)
    if os.environ.get("B200_PROFILE_TIMED"):
        torch.cuda.profiler.stop()
    launches = ops.LAUNCHES - l0
    timed_out = last["images"].clone() if args.dump_outputs else None  # the next calls reuse the pipeline's output buffers
    step_e2e()
    sec_e2e = timed(step_e2e, K)
    clk = clocks.stop()
    value = B * world * K / sec
    e2e_value = B * world * K / sec_e2e
    fam, fwd_ms, roof = {}, None, None
    if rank == 0:
        gf = next(iter(pipe._graphs.values()))
        s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s_.record()
        for _ in range(5):
            gf()
        e_.record()
        torch.cuda.synchronize()
        fwd_ms = s_.elapsed_time(e_) / 5
        ops.PROFILE = []
        gf._eager()
        torch.cuda.synchronize()
        for name, fl, by, s2, e2, *_ in ops.PROFILE:
            d = fam.setdefault(name, {"launches": 0, "flops": 0.0, "bytes": 0.0, "ms": 0.0})
            d["launches"] += 1
            d["flops"] += fl
            d["bytes"] += by
            d["ms"] += s2.elapsed_time(e2)
        ops.PROFILE = None
        for d in fam.values():
            d["tflops"] = d["flops"] / (d["ms"] * 1e-3) / 1e12 if d["ms"] > 0 else 0.0
            d["gbs"] = d["bytes"] / (d["ms"] * 1e-3) / 1e9 if d["ms"] > 0 else 0.0
        at = fam.get("attention", {"launches": 0, "flops": 0.0, "ms": 1.0})
        ach = at["flops"] / (at["ms"] * 1e-3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        roof = {"kernel": "b200::attn64s_kernel<DH=128> (small-CTA attention, joint txt+img attention, 24 heads x 128, 4352 tokens, batch %d)" % B,
                "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "peak_source": peaks["source"] + " (sustained: kernel timed inside a long step)", "launches": at["launches"],
                "avg_launch_ms": at["ms"] / max(1, at["launches"]), "flops_per_launch_avg": at["flops"] / max(1, at["launches"])}
        gflop = synthetic.FLUX_GFLOP_PER_SAMPLE
        line = {"metric": "images_per_sec_flux_dev_1024_euler_20steps_batch4", "value": value, "unit": UNIT, "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": sec / K * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16, fp32 accumulate and sampler state", "data": "synthetic",
                "config": {"workload": f"Flux.1-dev {args.size}x{args.size} txt2img (transformer + 16-channel VAE decode), Euler {S} steps, "
                                       f"Simple schedule, distilled guidance 3.5, batch {B}/GPU, {Lt} T5 tokens; 1 bench step = 1 batch",
                           "parallelism": f"replicas x{world} (request sharding by seed; NCCL gather of latents only)",
                           "l2": "working set (23.8 GB weights) >> 126 MB L2; no explicit flush"},
                "transformer_ms_per_step": fwd_ms,
                "transformer_roofline_ms_per_step": B * gflop * 1e9 / (peaks["bf16_tflops_sustained"] * 1e12) * 1e3,
                "flop_roofline_frac_whole_job": value / world * (S * gflop + synthetic.VAE_GFLOP_PER_IMAGE["sdxl@1024"] * (args.size / 1024) ** 2) * 1e9 / (peaks["bf16_tflops_sustained"] * 1e12),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": launches, "clocks": clk, "roofline": roof, "kernel_families": fam, "cpu_baseline": None}
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"images": timed_out})
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--sampler_steps", type=int, default=30)
    ap.add_argument("--workload", default="sdxl", choices=["sdxl", "sd15", "flux"],
                    help="sdxl = BASELINE.json's headline config (default); sd15 = configs[1]: SD1.5 512x512, Euler-a 20 steps, "
                         "batch 8; flux = configs[4]: Flux.1-dev 1024x1024, 20 steps, batch 4, bf16")
    ap.add_argument("--sampler", default="euler_a", choices=["euler_a", "dpmpp_2m"],
                    help="euler_a = the headline; dpmpp_2m = BASELINE.json configs[3] (DPM++ 2M, Karras schedule, run with --gpus 8)")
    ap.add_argument("--path", default="plugin", choices=["plugin", "pipeline"],
                    help="what `e2e` drives: plugin = the reference-facing plug points (P3 model_function_wrapper + P4 k-diffusion "
                         "sampler function + P5 VAE decode wrapper, called as Forge calls them); pipeline = Txt2ImgPipeline.generate")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (the decoded images [B, H, W, 3]; "
                         "under torchrun, the batch rank 0 computed itself) as DIR/images.npy, float32; above 64 MB a fixed, "
                         "seeded sample of its elements.  B200 arm only")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the B200 arm: the reference arm times UNet forwards, not whole jobs")

    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.workload == "flux":
        run_flux(args)
        return

    K = args.steps if args.steps is not None else 3
    W = args.warmup if args.warmup is not None else 3
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = torch.device("cuda", torch.cuda.current_device())

    from b200forge import dist as bdist
    from b200forge import k_samplers, lib, ops, plugin, synthetic
    from b200forge.pipeline import Txt2ImgPipeline
    lib.check(lib.load().b200_device_ok())
    peaks = load_peaks()

    sd15 = args.workload == "sd15"
    if sd15:  # BASELINE.json configs[1]
        if args.size == 1024:
            args.size = 512
        if args.sampler_steps == 30:
            args.sampler_steps = 20
    B, S = args.batch, args.sampler_steps
    hw = args.size // 8
    sampler = args.sampler
    cfg_scale = 7.0
    ucfg, vcfg = (synthetic.SD15, synthetic.VAE_SD15) if sd15 else (synthetic.SDXL, synthetic.VAE_SDXL)
    wl_name = "SD1.5" if sd15 else "SDXL-base"
    gflop_key = "sd15@64" if sd15 else "sdxl@128"
    unet_gflop = synthetic.UNET_GFLOP_PER_SAMPLE[gflop_key] * (hw * hw) / ((64 * 64) if sd15 else (128 * 128))
    vae_gflop = synthetic.VAE_GFLOP_PER_IMAGE["sdxl@1024"] * (args.size * args.size) / (1024 * 1024)  # same decoder architecture
    usd = synthetic.random_unet_state_dict(ucfg, device=dev, dtype=torch.float16, seed=0)
    vsd = synthetic.random_vae_decoder_state_dict(vcfg, device=dev, dtype=torch.bfloat16, seed=1)
    pipe = Txt2ImgPipeline(ucfg, usd, vae_cfg=vcfg, vae_state_dict=vsd, dtype=torch.float16, device=dev)
    del usd, vsd

    # ---- synthetic job inputs (pinned host copies for the e2e legs, device copies for the resident leg)
    seeds = bdist.shard_seeds(1000, B, rank, world)  # contiguous-by-seed sharding: results independent of N
    gens = [torch.Generator().manual_seed(sd_) for sd_ in seeds]

    def draw():
        return torch.stack([torch.randn((4, hw, hw), generator=g) for g in gens])

    g0 = torch.Generator().manual_seed(7)
    adm = ucfg["adm_in_channels"] or 8
    host = {
        "noise": draw().pin_memory(),
        "step_noise": torch.stack([draw() for _ in range(S - 1)]).pin_memory(),
        "cond": {"crossattn": torch.randn(B, 77, ucfg["context_dim"], generator=g0).half().pin_memory(),
                 "vector": torch.randn(B, adm, generator=g0).half().pin_memory()},
        "uncond": {"crossattn": torch.randn(B, 77, ucfg["context_dim"], generator=g0).half().pin_memory(),
                   "vector": torch.randn(B, adm, generator=g0).half().pin_memory()},
    }
    devin = {"noise": host["noise"].to(dev), "step_noise": host["step_noise"].to(dev),
             "cond": {k: v.to(dev) for k, v in host["cond"].items()},
             "uncond": {k: v.to(dev) for k, v in host["uncond"].items()}}
    uses_noise = sampler == "euler_a"
    h2d = (host["noise"].numel() * 4 + (host["step_noise"].numel() * 4 if uses_noise else 0) +
           sum(v.numel() * 2 for v in host["cond"].values()) + sum(v.numel() * 2 for v in host["uncond"].values()))
    out_host = torch.empty((B, args.size, args.size, 3), dtype=torch.float32).pin_memory()
    d2h = out_host.numel() * 4
    # multi-GPU: the only collective on the path — one gather of the finished images to rank 0, as uint8 (the conversion the
    # reference does on the host after its D2H copy): a quarter of the fp32 bytes
    gathered = [torch.empty((B, args.size, args.size, 3), dtype=torch.uint8, device=dev) for _ in range(world)] \
        if (dist is not None and rank == 0) else None

    def job(inp):
        return pipe.generate(inp["cond"], inp["uncond"], inp["noise"], steps=S, sampler=sampler, cfg_scale=cfg_scale,
                             step_noise=inp["step_noise"] if uses_noise else None)

    def finish(img):
        if dist is not None:
            bdist.gather_images_u8(img, bufs=gathered)

    # ---- the plug-in path: the same job driven exactly as Forge drives its backend (SURVEY 8b):
    #   CFGDenoiser.forward -> sampling_function_inner batches [uncond | cond] and calls model_options['model_function_wrapper']
    #   (P3, backend/sampling/sampling_function.py:270-273); the CFG combine stays in the caller's torch code (:292-322);
    #   k_diffusion.sampling.sample_* (P4) owns the loop; VAE.decode calls model_options['model_vae_decode_wrapper'] (P5).
    unet_w = plugin.UNetWrapper(pipe.unet, pipe.pred)
    vae_w = plugin.VAEDecodeWrapper(pipe.vae)
    has_y = pipe.unet.has_label
    sig_sched = None

    def plugin_job(inp):
        nonlocal sig_sched
        put = lambda t, dt: t.to(device=dev, dtype=dt, non_blocking=True)  # noqa: E731
        ctx = torch.cat([put(inp["uncond"]["crossattn"], torch.float16), put(inp["cond"]["crossattn"], torch.float16)])
        y = torch.cat([put(inp["uncond"]["vector"], torch.float16), put(inp["cond"]["vector"], torch.float16)]) if has_y else None
        noise = put(inp["noise"], torch.float32)
        sn = put(inp["step_noise"], torch.float32) if uses_noise else None
        if sig_sched is None:
            from b200forge import sampling as bs
            sig_sched = bs.make_sigmas(pipe.pred, sampler, S).to(dev)
        c = {"c_crossattn": ctx, "y": y, "transformer_options": {"cond_or_uncond": [1, 0]}}

        def unreachable(*a, **k):
            raise RuntimeError("the plug-in handed the call back to the reference path")

        def denoiser(x, sigma, **kw):  # sampling_function_inner for one cond + one uncond entry, both in one batch
            out = unet_w(unreachable, {"input": torch.cat([x, x]), "timestep": torch.cat([sigma, sigma]), "c": c,
                                       "cond_or_uncond": [1, 0]})
            un, co = out.chunk(2)
            return un + (co - un) * cfg_scale

        x0 = noise * sig_sched[0]  # predictor.noise_scaling(sigmas[0], noise, zeros, max_denoise=False)
        if sampler == "euler_a":
            it = iter(range(S))
            lat = k_samplers.sample_euler_ancestral(denoiser, x0, sig_sched, extra_args={}, disable=True,
                                                    noise_sampler=lambda s_, sn_: sn[next(it)])
        else:
            lat = k_samplers.sample_dpmpp_2m(denoiser, x0, sig_sched, extra_args={}, disable=True)
        # Forge hands P5 the processed-out latent (diffusion_engine/sdxl.py:134-138)
        return vae_w(unreachable, lat / pipe.vae.scaling), lat

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, iters):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(iters):
            fn()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) * 1e-3

    last = {}

    def step_resident():
        last["images"] = job(devin)
        finish(last["images"])

    def step_e2e_pipeline():
        img = job(host)
        finish(img)
        out_host.copy_(img, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the device->host read of the step's result

    def step_e2e_plugin():
        img, _ = plugin_job(host)
        finish(img)
        out_host.copy_(img, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    step_e2e = step_e2e_plugin if args.path == "plugin" else step_e2e_pipeline

    for _ in range(W):
        step_resident()
    clocks = ClockSampler(torch.cuda.current_device())
    clocks.start()
    l0 = ops.LAUNCHES
    if os.environ.get("B200_PROFILE_TIMED"):  # `ncu --profile-from-start off`: capture exactly the timed region
        torch.cuda.profiler.start()
    sec = timed(step_resident, K)
    if os.environ.get("B200_PROFILE_TIMED"):
        torch.cuda.profiler.stop()
    launches = ops.LAUNCHES - l0
    timed_out = last["images"].clone() if args.dump_outputs else None  # the next calls reuse the pipeline's output buffers
    step_e2e()  # untimed: graph capture / first-call setup of this leg
    l1 = ops.LAUNCHES
    sec_e2e = timed(step_e2e, K)
    launches_e2e = ops.LAUNCHES - l1
    other = step_e2e_pipeline if args.path == "plugin" else step_e2e_plugin
    other()
    sec_other = timed(other, K)
    clk = clocks.stop()

    total_images = B * world * K
    value = total_images / sec
    e2e_value = total_images / sec_e2e
    other_value = total_images / sec_other

    # ---- UNet ms/step and the per-kernel-family roofline from one instrumented eager denoise step + VAE decode
    unet_ms = None
    roof = None
    fam = {}
    if rank == 0:
        gu = next(iter(pipe._graphs.values()))
        s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        s_.record()
        for _ in range(10):
            gu()
        e_.record()
        torch.cuda.synchronize()
        unet_ms = s_.elapsed_time(e_) / 10
        ops.PROFILE = []
        gu._eager()
        pipe.decode(torch.randn(B, 4, hw, hw, device=dev) * 0.13025)
        torch.cuda.synchronize()
        for name, fl, by, s2, e2, *_ in ops.PROFILE:
            d = fam.setdefault(name, {"launches": 0, "flops": 0.0, "bytes": 0.0, "ms": 0.0})
            d["launches"] += 1
            d["flops"] += fl
            d["bytes"] += by
            d["ms"] += s2.elapsed_time(e2)
        ops.PROFILE = None
        tens = {"launches": 0, "flops": 0.0, "ms": 0.0}
        for name in ("gemm", "conv3x3"):
            if name in fam:
                for k in tens:
                    tens[k] += fam[name][k]
        ach = tens["flops"] / (tens["ms"] * 1e-3) / 1e12 if tens["ms"] > 0 else 0.0
        peak = peaks["bf16_tflops_sustained"]
        roof = {"kernel": "b200::gemm_kernel (tcgen05 GEMM + implicit-GEMM conv3x3; 1 UNet forward @batch 16 + VAE decode)",
                "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                # not measured in this run (ncu cannot wrap a timed run); per-kernel dram bytes from the committed
                # `ncu --set full` captures are in profiles/ncu_r2_summary.md
                "traffic": None,
                "peak_source": peaks["source"] + " (sustained: kernel timed inside a long step)",
                "launches": tens["launches"], "avg_launch_ms": tens["ms"] / max(1, tens["launches"]),
                "flops_per_launch_avg": tens["flops"] / max(1, tens["launches"])}
        for name, d in fam.items():
            d["tflops"] = d["flops"] / (d["ms"] * 1e-3) / 1e12 if d["ms"] > 0 else 0.0
            d["gbs"] = d["bytes"] / (d["ms"] * 1e-3) / 1e9 if d["ms"] > 0 else 0.0

    # ---- parity at the benchmarked shape, in the same process, after the timed region (rank 0, N = 1)
    cpu_base = None
    gpu_ref = None
    parity = None
    attn_pair = None
    if rank == 0 and world == 1:
        img_chk, lat_plugin = plugin_job(devin)
        lat_pipe = pipe.sample(devin["cond"], devin["uncond"], devin["noise"], steps=S, sampler=sampler, cfg_scale=cfg_scale,
                               step_noise=devin["step_noise"] if uses_noise else None)
        torch.cuda.synchronize()
        finite = bool(torch.isfinite(lat_pipe).all() and torch.isfinite(lat_plugin).all() and torch.isfinite(img_chk).all())
        if not finite:
            print(json.dumps({"error": "non-finite output at the benchmarked shape", "metric": METRIC}), flush=True)
            sys.exit(1)

        def psnr(a, b):
            mse = (a.float() - b.float()).pow(2).mean()
            return float(10 * torch.log10(b.float().abs().max() ** 2 / mse.clamp_min(1e-30)))

        parity = {"finite": True,
                  "plugin_vs_pipeline_final_latent": {"psnr_db": psnr(lat_plugin, lat_pipe),
                                                      "rel_rms": float((lat_plugin - lat_pipe).pow(2).mean().sqrt() / lat_pipe.pow(2).mean().sqrt())}}
        if not args.no_parity:
            parity["unet_forward_vs_oracle_fp32"] = unet_forward_parity(pipe, ucfg, hw, 2 * B, dev)
        if not args.no_gpu_reference:
            try:
                attn_pair = attention_vs_sdpa(dev)
                gpu_ref, lat_ref = gpu_reference_job(ucfg, vcfg, B, S, hw, devin["cond"], devin["uncond"], devin["noise"],
                                                     devin["step_noise"], sampler, cfg_scale)
                parity["final_latent_vs_reference_fp16_loop"] = {
                    "psnr_db": psnr(lat_pipe, lat_ref), "steps": S, "sampler": sampler,
                    "rel_rms": float((lat_pipe - lat_ref).pow(2).mean().sqrt() / lat_ref.pow(2).mean().sqrt()),
                    "what": "same seeds / injected noise; ours = fused fp16 pipeline, reference = oracle-port loop in fp16 on this GPU"}
                # short horizon: rounding differences have not yet been amplified by the (random-weight) UNet
                _, lat_ref4 = gpu_reference_job(ucfg, vcfg, B, S, hw, devin["cond"], devin["uncond"], devin["noise"],
                                                devin["step_noise"], sampler, cfg_scale, max_steps=4)
                from b200forge import sampling as bs
                sig4 = bs.make_sigmas(pipe.pred, sampler, S)[:5]
                lat4 = pipe.sample(devin["cond"], devin["uncond"], devin["noise"], steps=4, sampler=sampler, cfg_scale=cfg_scale,
                                   sigmas=sig4, step_noise=devin["step_noise"] if uses_noise else None)
                parity["first_4_steps_vs_reference_fp16_loop"] = {
                    "psnr_db": psnr(lat4, lat_ref4),
                    "rel_rms": float((lat4 - lat_ref4).pow(2).mean().sqrt() / lat_ref4.pow(2).mean().sqrt())}
            except Exception as ex:  # context numbers only
                gpu_ref = {"failed": f"{type(ex).__name__}: {ex}"}
        if not args.no_cpu_baseline and not sd15:
            threads = usable_cores()
            fwd = cpu_baseline_sample(hw, threads)
            t = fwd()
            cpu_base = {"value": images_per_sec_from_forward(t, S), "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": (f"1 SDXL UNet sample-forward (batch 1, latent {hw}x{hw}, fp32 ATen via the oracle port) "
                                   f"= {t:.2f} s; images/s = 1/(2*{S}*t), VAE decode excluded")}

    if rank == 0:
        flops_per_image = 2 * S * unet_gflop * 1e9 + vae_gflop * 1e9
        samp_name = {"euler_a": "Euler-a", "dpmpp_2m": "DPM++ 2M (Karras)"}[sampler]
        metric = METRIC if (not sd15 and sampler == "euler_a") else \
            f"images_per_sec_{'sd15' if sd15 else 'sdxl'}_{args.size}_{sampler}_{S}steps_batch{B}"
        e2e_name = {"plugin": "plug points P3 (model_function_wrapper) + P4 (k_diffusion sample_*) + P5 (VAE decode wrapper), CFG combine "
                              "in the caller's torch code as in Forge",
                    "pipeline": "Txt2ImgPipeline.generate (one-launch CFG + sampler step)"}
        line = {
            "metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": sec / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16 (UNet) / bf16 (VAE), fp32 accumulate and sampler state", "data": "synthetic",
            "config": {"workload": f"{wl_name} {args.size}x{args.size} txt2img, {samp_name} {S} steps, CFG 7, batch {B}/GPU "
                                   f"(UNet batch {2 * B}), VAE decode included; 1 bench step = 1 batch of {B} images/GPU",
                       "parallelism": f"replicas x{world} (request sharding by seed; NCCL gather of uint8 images only)",
                       "l2": "working set (5.1 GB weights + activations) >> 126 MB L2; no explicit flush",
                       "roofline_pass": "separate instrumented eager pass after the timed region (graph replays cannot be bracketed)",
                       "e2e_path": args.path + ": " + e2e_name[args.path]},
            "unet_ms_per_step": unet_ms,
            "unet_roofline_ms_per_step": 2 * B * unet_gflop * 1e9 / (peaks["bf16_tflops_sustained"] * 1e12) * 1e3,
            "flop_roofline_frac_whole_job": value / world * flops_per_image / (peaks["bf16_tflops_sustained"] * 1e12),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "path": args.path,
                    "gpu_launches": launches_e2e},
            "e2e_other_path": {"value": other_value, "unit": UNIT, "path": "pipeline" if args.path == "plugin" else "plugin"},
            "gpu_launches": launches,
            "clocks": clk,
            "roofline": roof,
            "kernel_families": fam,
            "parity": parity,
            "cpu_baseline": cpu_base,
            "gpu_reference": gpu_ref,
            "gpu_reference_unet_ms_per_step": None if not isinstance(gpu_ref, dict) else gpu_ref.get("unet_ms_per_step"),
            "attention_vs_sdpa": attn_pair,
        }
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"images": timed_out})
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
