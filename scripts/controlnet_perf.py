"""ControlNet cost at the SDXL 1024^2 working point: batch 8 images x [uncond | cond] = 16 rows, latent 128x128, one hint
image [1, 3, 1024, 1024], full-width SDXL ControlNet (oracle.controlnet.SDXL_CONTROLNET) with seeded random weights.

    python scripts/controlnet_perf.py [--out profiles/controlnet_perf_b200.json] [--iters 20]

Reports, with the card's name and power limit read in the same run:
  controlnet_ms          fused ControlNetEngine.forward per call (guided hint cached, as from the second step of a job on)
  port_ms                the oracle port in fp16 (torch: cuDNN convolutions, SDPA attention) on the same inputs, same process,
                         as the reference runs it: input_hint_block on the 1024^2 hint in every call
  port_ms_hint_cached    the same port with the hint block computed once beforehand (like for like with controlnet_ms)
  tflop / family_ms      algorithmic FLOP of one forward and per-family kernel time (ops.PROFILE instrumented pass); the
                         layout / elementwise launches that ops.PROFILE does not bracket (NCHW <-> NHWC conversions, im2col of
                         conv_in and the stride-2 downsamples, the guided-hint add, time embedding, SiLU) are bracketed here
                         as family "layout+elementwise"; unaccounted_ms = controlnet_ms - their sum (gaps between launches)
  guided_hint_ms         input_hint_block on the one hint image (once per job)
  step_ms                one sampler step through the plug points: UNet alone (P3) vs ControlNet (P6) + UNet (P3)
  batch2_host_ms / _gpu  host enqueue time vs device time of a batch-2 ControlNet call (is the eager path host-bound?);
                         batch2_host_ms_p6 the same call enqueued through the P6 wrapper
Timings are CUDA events over >= `--iters` calls after warm-up; the working set (weights ~2.5 GB + activations) exceeds L2.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from b200forge import ops, plugin  # noqa: E402
from b200forge.controlnet_engine import ControlNetEngine  # noqa: E402
from b200forge.unet_engine import UNetEngine  # noqa: E402
from oracle import configs as CF  # noqa: E402
from oracle import controlnet as OC  # noqa: E402
from oracle import sampling as S  # noqa: E402
from oracle import unet as OU  # noqa: E402

DEV = "cuda"


def timed(fn, iters):
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


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "controlnet_perf_b200.json"))
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("controlnet_perf.py measures on the GPU; no CUDA device")
    res = {"card": card(), "shape": "SDXL ControlNet, x [16,4,128,128], hint [1,3,1024,1024], fp16"}
    ccfg = OC.SDXL_CONTROLNET
    csd = {k: v.half() for k, v in OC.random_controlnet_state_dict(ccfg, 3, seed=21).items()}
    eng = ControlNetEngine(ccfg, csd, dtype=torch.float16, device=DEV)
    g = torch.Generator().manual_seed(22)
    n = 16
    x = torch.randn(n, 4, 128, 128, generator=g).half().to(DEV)
    hint = torch.rand(1, 3, 1024, 1024, generator=g).half().to(DEV)
    ctx = torch.randn(n, 77, ccfg["context_dim"], generator=g).half().to(DEV)
    y = torch.randn(n, ccfg["adm_in_channels"], generator=g).half().to(DEV)
    t = torch.linspace(999.0, 1.0, n, device=DEV)

    # 1. ours vs the fp16 port
    res["controlnet_ms"] = timed(lambda: eng.forward(x, hint, t, ctx, y), a.iters)
    sd16 = {k: v.to(DEV) for k, v in csd.items()}
    with torch.no_grad():
        res["port_ms"] = timed(lambda: OC.controlnet_forward(sd16, ccfg, x, hint, t, ctx, y), a.iters)
        gh16 = OC.hint_block(sd16, ccfg, hint, x.dtype)
        res["port_ms_hint_cached"] = timed(lambda: OC.controlnet_forward(sd16, ccfg, x, hint, t, ctx, y, guided_hint=gh16),
                                           a.iters)
    res["ratio_ours_over_port"] = res["controlnet_ms"] / res["port_ms"]
    res["ratio_ours_over_port_hint_cached"] = res["controlnet_ms"] / res["port_ms_hint_cached"]
    res["target_ratio"] = 0.65
    res["target_met"] = res["ratio_ours_over_port"] <= 0.65
    del sd16, gh16

    # 2. algorithmic FLOP and per-family time (instrumented pass: every call bracketed by events)
    def bracketed(fn):
        def call(*args, **kw):
            with ops._prof("layout+elementwise"):
                return fn(*args, **kw)
        return call

    unbracketed = ("im2col3x3", "nchw_to_nhwc", "nhwc_to_nchw", "add_control_", "timestep_embedding", "silu")
    saved = {k: getattr(ops, k) for k in unbracketed}
    for k in unbracketed:
        setattr(ops, k, bracketed(saved[k]))
    ops.PROFILE = []
    eng.forward(x, hint, t, ctx, y)
    torch.cuda.synchronize()
    fam, flops = {}, 0.0
    for name, fl, by, s2, e2, *_ in ops.PROFILE:
        fam[name] = fam.get(name, 0.0) + s2.elapsed_time(e2)
        flops += fl
    ops.PROFILE = None
    for k, fn in saved.items():
        setattr(ops, k, fn)
    res["tflop"] = flops / 1e12
    res["family_ms"] = fam
    res["unaccounted_ms"] = res["controlnet_ms"] - sum(fam.values())
    res["achieved_tflops"] = flops / 1e12 / (res["controlnet_ms"] / 1e3)

    # 3. guided hint, once per job
    def hint_once():
        eng._hints.clear()
        eng.guided_hint(hint)
    res["guided_hint_ms"] = timed(hint_once, 5)
    eng.guided_hint(hint)

    # 4. one sampler step through the plug points: UNet alone vs ControlNet (P6) + UNet (P3)
    ucfg = CF.SDXL
    usd = {k: v.half() for k, v in OU.random_state_dict(ucfg, seed=11).items()}
    ueng = UNetEngine(ucfg, usd, dtype=torch.float16, device=DEV)
    del usd

    class P:
        prediction_type = "epsilon"
        timestep = staticmethod(lambda s: S.EpsPrediction().timestep(s.cpu()).to(s.device))

    pw = plugin.UNetWrapper(ueng, P())
    cw = plugin.ControlNetWrapper()

    class Inner:  # cldm.ControlNet as the wrapper sees it; never called (the fused path serves every call here)
        model_channels, num_res_blocks, channel_mult = ccfg["model_channels"], ccfg["num_res_blocks"], ccfg["channel_mult"]
        num_heads, num_head_channels = ccfg["num_heads"], ccfg["num_head_channels"]

        def state_dict(self):
            return csd

        def modules(self):
            return iter([self])

    class Unit:
        device = torch.device(DEV)

    inner = Inner()
    xl = torch.randn(n, 4, 128, 128, generator=g).to(DEV) * 3
    sig = torch.full((n,), 3.0, device=DEV)
    ctx32, y32 = ctx.float(), y.float()
    tt = P.timestep(sig).float()
    xc = S.EpsPrediction().calculate_input(sig.cpu(), xl.cpu()).to(DEV).half()

    def step_unet():
        c = {"c_crossattn": ctx32, "y": y32, "transformer_options": {}}
        return pw(None, {"input": xl, "timestep": sig, "c": c, "cond_or_uncond": [1, 0]})

    def step_cn():
        outs = cw(x=xc, hint=hint, timesteps=tt, context=ctx, y=y, model=Unit(), inner_model=inner)
        ctrl = {"input": [], "middle": [outs[-1] * 0.8], "output": [o * 0.8 for o in outs[:-1]]}
        c = {"c_crossattn": ctx32, "y": y32, "control": ctrl, "transformer_options": {}}
        return pw(None, {"input": xl, "timestep": sig, "c": c, "cond_or_uncond": [1, 0]})

    res["step_ms_unet_p3"] = timed(step_unet, a.iters)
    res["step_ms_controlnet_p6_plus_unet_p3"] = timed(step_cn, a.iters)
    res["plug_calls"] = {"p3_fast": pw.calls_fast, "p3_reference": pw.calls_reference, "p6_fast": cw.calls_fast,
                         "p6_reference": cw.calls_reference}

    # 5. host launch time vs GPU time of a batch-2 ControlNet call
    x2, ctx2, y2, t2 = x[:2].contiguous(), ctx[:2].contiguous(), y[:2].contiguous(), t[:2].contiguous()
    res["batch2_gpu_ms"] = timed(lambda: eng.forward(x2, hint, t2, ctx2, y2), a.iters)
    torch.cuda.synchronize()
    host = []
    for _ in range(a.iters):
        h0 = time.perf_counter()
        eng.forward(x2, hint, t2, ctx2, y2)
        host.append((time.perf_counter() - h0) * 1e3)
        torch.cuda.synchronize()
    res["batch2_host_ms"] = sorted(host)[len(host) // 2]
    host = []
    for _ in range(a.iters):
        h0 = time.perf_counter()
        cw(x=x2, hint=hint, timesteps=t2, context=ctx2, y=y2, model=Unit(), inner_model=inner)
        host.append((time.perf_counter() - h0) * 1e3)
        torch.cuda.synchronize()
    res["batch2_host_ms_p6"] = sorted(host)[len(host) // 2]
    n0 = ops.LAUNCHES
    eng.forward(x2, hint, t2, ctx2, y2)
    res["batch2_launches"] = ops.LAUNCHES - n0
    torch.cuda.synchronize()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
