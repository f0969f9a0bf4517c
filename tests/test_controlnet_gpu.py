"""GPU tests of the ControlNet path: the broadcasting control-add kernel, the fused ControlNet forward (ControlNetEngine)
against the reference goldens and the fp32 oracle at full width, the P6 plug point shared by two ControlNet units, and an
end-to-end Euler-a loop ControlNet (P6) -> control_merge -> UNet (P3).

Tolerances as for the UNet (SURVEY §8d): fp16 engine vs fp32 reference rel-RMS <= 3e-3, max-abs <= 2e-2 of the output's
RMS at full width (4e-2 absolute on the unit-scale goldens); final latent PSNR >= 40 dB."""
import pytest
import torch

from oracle import configs as CF
from oracle import controlnet as OC
from oracle import sampling as S
from oracle import unet as OU
from oracle.gen_controlnet_golden import make_inputs
from oracle.golden import load_golden
from tests.util import assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("nhwc", [False, True])
@pytest.mark.parametrize("batch1", [False, True])
@pytest.mark.parametrize("ctrl_f32", [True, False])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_add_control_kernel(nhwc, batch1, ctrl_f32, dtype):
    from b200forge import ops
    g = torch.Generator().manual_seed(4)
    n, hh, ww, c = 3, 12, 20, 200
    h = torch.randn(n, hh, ww, c, generator=g).to(dtype).to(DEV)
    shp = (1 if batch1 else n,) + ((hh, ww, c) if nhwc else (c, hh, ww))
    ctrl = torch.randn(*shp, generator=g).to(torch.float32 if ctrl_f32 else dtype).to(DEV)
    ref = h.float() + (ctrl.float() if nhwc else ctrl.float().permute(0, 2, 3, 1))
    ops.add_control_(h, ctrl, nhwc=nhwc)
    torch.cuda.synchronize()
    # one rounding of |h + ctrl| < 8 to the activation dtype: half an ulp is 2^-8 in fp16, 2^-5 in bf16
    assert_close(f"add_control nhwc={nhwc} batch1={batch1} ctrl_f32={ctrl_f32} {dtype}", h, ref,
                 max_abs=4e-3 if dtype == torch.float16 else 3.2e-2)


class _P:  # the two things UNetWrapper reads from Forge's predictor
    prediction_type = "epsilon"
    timestep = staticmethod(lambda s: S.EpsPrediction().timestep(s.cpu()).to(s.device))


def test_p3_t2i_batch1_residuals_vs_oracle():
    """T2I-Adapter residuals computed from one hint image have batch 1 (broadcast_image_to, controlnet.py:153-156): the
    fused UNet adds them to every image, as the reference's `h += ctrl` does."""
    from b200forge import plugin
    from b200forge.unet_engine import UNetEngine
    g = load_golden("unet_tiny_xl_control.pt")
    cfg = CF.CONFIGS["tiny_xl"]
    sd = OU.random_state_dict(cfg, seed=1)
    w = plugin.UNetWrapper(UNetEngine(cfg, sd, dtype=torch.float16, device=DEV), _P())
    ctrl1 = {k: [None if t is None else t[:1].to(DEV) for t in lst] for k, lst in g["control"].items()}
    x = (g["x"] * 5).to(DEV)
    sigma = torch.tensor([6.0, 0.8], device=DEV)
    c = {"c_crossattn": g["context"].to(DEV), "y": g["y"].to(DEV), "control": ctrl1, "transformer_options": {}}
    out = w(lambda *a, **k: None, {"input": x, "timestep": sigma, "c": c, "cond_or_uncond": [1, 0]})
    assert w.calls_fast == 1
    pred = S.EpsPrediction()
    ctrl_cpu = {k: [None if t is None else t.cpu() for t in lst] for k, lst in ctrl1.items()}
    with torch.no_grad():
        xc = pred.calculate_input(sigma.cpu(), x.cpu())
        eps = OU.unet_forward(sd, cfg, xc, pred.timestep(sigma.cpu()).float(), g["context"], g["y"], control=ctrl_cpu)
        ref = pred.calculate_denoised(sigma.cpu(), eps, x.cpu())
    assert_close("P3 + batch-1 T2I residuals vs oracle", out, ref, rel_rms=3e-3)


@pytest.mark.parametrize("name", ["tiny_xl", "tiny_15h"])
@pytest.mark.parametrize("hint", ["hint1", "hintN"])
def test_engine_vs_reference_golden(name, hint):
    from b200forge.controlnet_engine import ControlNetEngine
    g = load_golden(f"controlnet_{name}.pt")
    cfg = OC.CONFIGS[name]
    sd = OC.random_controlnet_state_dict(cfg, cfg["hint_channels"], seed=g["weight_seed"])
    v = make_inputs(g["shapes"], g["input_seed"])
    eng = ControlNetEngine(cfg, sd, dtype=torch.float16, device=DEV)
    y = v.get("y")
    outs = eng.forward(v["x"].half().to(DEV), v[hint].half().to(DEV), v["t"].to(DEV), v["context"].half().to(DEV),
                       None if y is None else y.half().to(DEV))
    torch.cuda.synchronize()
    for i, (o, r) in enumerate(zip(outs, g["out"][hint])):
        assert o.dtype == torch.float16 and o.is_contiguous()
        assert_close(f"controlnet {name} {hint} fp16 engine vs reference golden, out {i}", o, r, rel_rms=3e-3, max_abs=4e-2)


@pytest.mark.parametrize("name,hh,ww", [("sdxl", 128, 128), ("sd15", 64, 64), ("sdxl", 152, 104)])
def test_full_width_vs_oracle_fp32(name, hh, ww):
    """Full-size ControlNet at batch 16 (8 images x [uncond | cond]) with one 8x hint image, against the oracle in fp32 on
    the GPU (TF32 off) with the same fp16-rounded weights; two runs bit-identical."""
    from b200forge.controlnet_engine import ControlNetEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = OC.CONFIGS[name]
    sd = {k: v.half() for k, v in OC.random_controlnet_state_dict(cfg, 3, seed=21).items()}
    eng = ControlNetEngine(cfg, sd, dtype=torch.float16, device=DEV)
    g = torch.Generator().manual_seed(22)
    n = 16
    x = torch.randn(n, 4, hh, ww, generator=g).half().to(DEV)
    hint = torch.rand(1, 3, 8 * hh, 8 * ww, generator=g).half().to(DEV)
    ctx = torch.randn(n, 77, cfg["context_dim"], generator=g).half().to(DEV)
    y = torch.randn(n, cfg["adm_in_channels"], generator=g).half().to(DEV) if cfg["adm_in_channels"] else None
    t = torch.linspace(999.0, 1.0, n, device=DEV)
    outs = eng.forward(x, hint, t, ctx, y)
    eng._hints.clear()  # the second run recomputes the hint block too
    outs2 = eng.forward(x, hint, t, ctx, y)
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(outs, outs2)), "two runs differ"
    del outs2
    sd32 = {k: v.float().to(DEV) for k, v in sd.items()}
    with torch.no_grad():
        ref = OC.controlnet_forward(sd32, cfg, x.float(), hint.float(), t, ctx.float(), None if y is None else y.float())
    for i, (o, r) in enumerate(zip(outs, ref)):
        assert_close(f"controlnet {name} {hh}x{ww} full width fp16 engine vs oracle fp32, out {i}", o, r,
                     max_rel=2e-2, rel_rms=3e-3)


@pytest.mark.parametrize("name", ["tiny_xl_noattn", "tiny_xl_noattn_nomid"])
def test_engine_without_cross_attention_vs_oracle(name):
    """Every transformer depth 0 (the middle block's SpatialTransformer of depth 0, or none): GroupNorm + proj_in +
    proj_out only, against the oracle in fp32 on the same fp16-rounded weights."""
    from b200forge.controlnet_engine import ControlNetEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = OC.CONFIGS[name]
    sd = {k: v.half() for k, v in OC.random_controlnet_state_dict(cfg, 3, seed=5).items()}
    eng = ControlNetEngine(cfg, sd, dtype=torch.float16, device=DEV)
    g = torch.Generator().manual_seed(6)
    x = torch.randn(4, 4, 32, 32, generator=g).half().to(DEV)
    hint = torch.rand(1, 3, 256, 256, generator=g).half().to(DEV)
    ctx = torch.randn(4, 77, cfg["context_dim"], generator=g).half().to(DEV)
    y = torch.randn(4, cfg["adm_in_channels"], generator=g).half().to(DEV)
    t = torch.tensor([900.0, 500.0, 100.0, 5.0], device=DEV)
    outs = eng.forward(x, hint, t, ctx, y)
    sd32 = {k: v.float().to(DEV) for k, v in sd.items()}
    with torch.no_grad():
        ref = OC.controlnet_forward(sd32, cfg, x.float(), hint.float(), t, ctx.float(), y.float())
    for i, (o, r) in enumerate(zip(outs, ref)):
        assert_close(f"controlnet {name} fp16 engine vs oracle fp32, out {i}", o, r, max_rel=2e-2, rel_rms=3e-3)


class _StandIn:
    """cldm.ControlNet as the P6 wrapper sees it (constructor attributes, state_dict, modules, call)."""

    def __init__(self, cfg, sd):
        self.cfg, self.sd = cfg, sd
        self.model_channels, self.num_res_blocks, self.channel_mult = cfg["model_channels"], cfg["num_res_blocks"], cfg["channel_mult"]
        self.num_heads, self.num_head_channels = cfg["num_heads"], cfg["num_head_channels"]

    def state_dict(self):
        return self.sd

    def modules(self):
        return iter([self])

    def __call__(self, x, hint, timesteps, context, y=None):
        with torch.no_grad():
            return OC.controlnet_forward(self.sd, self.cfg, x.float(), hint.float(), timesteps, context.float(),
                                         None if y is None else y.float())


class _Unit:  # backend.patcher.controlnet.ControlNet, as far as the wrapper looks at it
    device = torch.device(DEV)


def _control_merge(outs, strength, output_dtype):
    """ControlBase.control_merge (controlnet.py:230-279) for one ControlNet without weighting or masks."""
    out = {"input": [], "middle": [], "output": []}
    for i, x in enumerate(outs):
        x *= strength
        out["middle" if i == len(outs) - 1 else "output"].append(x.to(output_dtype))
    return out


def test_p6_two_units_share_one_model():
    from b200forge import plugin
    cfg = OC.CONFIGS["tiny_xl"]
    sd = OC.random_controlnet_state_dict(cfg, 3, seed=31)
    inner = _StandIn(cfg, {k: v.to(DEV) for k, v in sd.items()})
    w = plugin.ControlNetWrapper()
    g = torch.Generator().manual_seed(32)
    x = torch.randn(4, 4, 16, 16, generator=g).half().to(DEV)
    ctx = torch.randn(4, 77, cfg["context_dim"], generator=g).half().to(DEV)
    y = torch.randn(4, cfg["adm_in_channels"], generator=g).half().to(DEV)
    t = torch.tensor([900.0, 900.0, 300.0, 300.0], device=DEV)
    hints = [torch.rand(1, 3, 128, 128, generator=g).half().to(DEV) for _ in range(2)]
    for rep in range(2):  # the second round is served from the guided-hint cache
        for hint in hints:
            outs = w(x=x, hint=hint, timesteps=t, context=ctx, y=y, model=_Unit(), inner_model=inner)
            ref = inner(x, hint, t, ctx, y)
            for i, (o, r) in enumerate(zip(outs, ref)):
                assert_close(f"P6 shared model, round {rep}, out {i}", o, r, rel_rms=3e-3, max_rel=2e-2)
    assert len(w.engines) == 1 and w.calls_fast == 4 and w.calls_reference == 0


def test_end_to_end_euler_a_controlnet_p6_p3():
    """6 Euler-a steps with CFG on the tiny SDXL topology: each step the ControlNet runs through P6 on the [uncond | cond]
    batch, a stand-in for get_control / control_merge scales its outputs (strength 0.8) into the "output" / "middle" lists,
    and the UNet adds them through P3.  Compared with the same loop on the oracle in fp32."""
    from b200forge import plugin
    from b200forge.unet_engine import UNetEngine
    cfg, ccfg = CF.CONFIGS["tiny_xl"], OC.CONFIGS["tiny_xl"]
    usd = OU.random_state_dict(cfg, seed=1)
    csd = OC.random_controlnet_state_dict(ccfg, 3, seed=41)
    pw = plugin.UNetWrapper(UNetEngine(cfg, usd, dtype=torch.float16, device=DEV), _P())
    cw = plugin.ControlNetWrapper()
    inner = _StandIn(ccfg, {k: v.to(DEV) for k, v in csd.items()})
    pred = S.EpsPrediction()
    g = torch.Generator().manual_seed(42)
    B, steps, cfg_scale, strength = 2, 6, 5.0, 0.8
    cond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g), vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    uncond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g), vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    hint = torch.rand(1, 3, 128, 128, generator=g)
    noise = torch.randn(B, 4, 16, 16, generator=g)
    step_noise = torch.randn(steps, B, 4, 16, 16, generator=g)
    sigmas = S.get_sigmas_uniform(pred, steps)
    ctx = torch.cat([uncond["crossattn"], cond["crossattn"]])
    yv = torch.cat([uncond["vector"], cond["vector"]])

    def fast(x, sigma):
        xin, sig = torch.cat([x, x]), torch.cat([sigma, sigma])
        xc = pred.calculate_input(sig.cpu(), xin.cpu()).to(DEV)
        tt = pred.timestep(sig.cpu()).float().to(DEV)
        outs = cw(x=xc.half(), hint=hint_dev, timesteps=tt, context=ctx.to(DEV).half(), y=yv.to(DEV).half(),
                  model=_Unit(), inner_model=inner)
        c = {"c_crossattn": ctx.to(DEV), "y": yv.to(DEV), "control": _control_merge(outs, strength, torch.float32),
             "transformer_options": {}}
        den = pw(lambda *a, **k: None, {"input": xin, "timestep": sig, "c": c, "cond_or_uncond": [1, 0]})
        u, cc = den.chunk(2)
        return u + (cc - u) * cfg_scale

    def oracle(x, sigma):
        xin, sig = torch.cat([x, x]), torch.cat([sigma, sigma])
        xc = pred.calculate_input(sig, xin)
        tt = pred.timestep(sig).float()
        outs = OC.controlnet_forward(csd, ccfg, xc, hint, tt, ctx, yv)
        eps = OU.unet_forward(usd, cfg, xc, tt, ctx, yv, control=_control_merge(outs, strength, torch.float32))
        den = pred.calculate_denoised(sig, eps, xin)
        u, cc = den.chunk(2)
        return u + (cc - u) * cfg_scale

    hint_dev = hint.half().to(DEV)
    x0 = pred.noise_scaling(sigmas[0], noise.clone(), torch.zeros_like(noise), max_denoise=False)
    k1, k2 = iter(range(steps)), iter(range(steps))
    out = S.sample_euler_ancestral(fast, x0.to(DEV), sigmas.to(DEV), lambda: step_noise[next(k1)].to(DEV))
    with torch.no_grad():
        ref = S.sample_euler_ancestral(oracle, x0, sigmas, lambda: step_noise[next(k2)])
    torch.cuda.synchronize()
    assert cw.calls_fast == steps and pw.calls_fast == steps and pw.calls_reference == 0
    mse = (out.cpu() - ref).pow(2).mean().item()
    psnr = 10 * torch.log10(torch.tensor((ref.max() - ref.min()).item() ** 2 / max(mse, 1e-30))).item()
    print(f"[parity] ControlNet + UNet Euler-a 6 steps: latent PSNR {psnr:.1f} dB")
    assert psnr >= 40.0, psnr
