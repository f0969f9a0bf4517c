"""First hardware runs of everything round 1 shipped on CPU emulation only (VERDICT r1, "weak" 4 / "next" 2):
`b200_add_nchw` + ControlNet residuals, `b200_rmsnorm_rows` + ChromaEngine, the LMS / SDE sampler plans, hires-fix, the
v-prediction pipeline, the non-tiling-size routes at a real SDXL bucket (1216x832 -> 152x104 latents), plus the ADVICE fixes
that touch device code (GEMM alpha / scaled logits, sampler_update argument handling)."""
import os

import pytest
import torch

from oracle import configs as CF
from oracle import ops as O
from oracle import sampling as S
from oracle import unet as OU
from oracle import vae as OV
from tests.util import assert_close, err_stats

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _gold(name):
    from oracle.golden import load_golden
    return load_golden(name)


def _rand(*shape, dtype=torch.float16, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dtype).to(DEV)


# ------------------------------------------------------------------------------------------------ f3: control residuals
@pytest.mark.parametrize("ctrl_dtype", [torch.float16, torch.float32])
def test_add_nchw(ctrl_dtype):
    from b200forge import ops
    n, h, w, c = 3, 24, 40, 320
    x = _rand(n, h, w, c, seed=1)
    ctrl = _rand(n, c, h, w, seed=2).to(ctrl_dtype)
    ref = (x.float() + ctrl.float().permute(0, 2, 3, 1)).half()
    ops.add_nchw_(x, ctrl)
    torch.cuda.synchronize()
    assert_close(f"add_nchw {ctrl_dtype}", x, ref.float(), max_abs=2e-3)


def test_unet_control_residuals_vs_reference_golden():
    """ControlNet / T2I-Adapter residuals consumed inside the fused forward (backend/nn/unet.py:44-52, 714, 733, 739) against
    the imported reference's output with the same synthetic residuals."""
    from b200forge.unet_engine import UNetEngine
    g = _gold("unet_tiny_xl_control.pt")
    cfg = CF.CONFIGS[g["config"]]
    sd = OU.random_state_dict(cfg, seed=g["weight_seed"])
    eng = UNetEngine(cfg, sd, dtype=torch.float16, device=DEV)
    control = {k: [None if t is None else t.to(DEV) for t in v] for k, v in g["control"].items()}
    out = eng.forward(g["x"].to(DEV).half(), g["t"].to(DEV), g["context"].to(DEV).half(), g["y"].to(DEV).half(), control=control)
    plain = eng.forward(g["x"].to(DEV).half(), g["t"].to(DEV), g["context"].to(DEV).half(), g["y"].to(DEV).half())
    torch.cuda.synchronize()
    assert_close("unet + control residuals vs reference golden", out, g["out"], max_abs=4e-2, rel_rms=3e-3)
    assert err_stats(plain, g["out"])[1] > 5e-2, "the residuals must matter in this fixture"
    assert all(len(v) == len(g["control"][k]) for k, v in control.items()), "the caller's lists stay intact"


def test_p3_wrapper_passes_control_on_device():
    from b200forge import plugin
    from b200forge.unet_engine import UNetEngine
    g = _gold("unet_tiny_xl_control.pt")
    cfg = CF.CONFIGS[g["config"]]
    sd = OU.random_state_dict(cfg, seed=g["weight_seed"])
    eng = UNetEngine(cfg, sd, dtype=torch.float16, device=DEV)
    pred = S.EpsPrediction()

    class P:
        prediction_type = "epsilon"
        timestep = staticmethod(lambda s: pred.timestep(s))

    w = plugin.UNetWrapper(eng, P())
    x = (torch.randn(2, 4, 16, 16, generator=torch.Generator().manual_seed(3)) * 3).to(DEV)
    sigma = torch.tensor([4.0, 0.5], device=DEV)
    control = {k: [None if t is None else t.to(DEV) for t in v] for k, v in g["control"].items()}
    c = {"c_crossattn": g["context"].to(DEV), "y": g["y"].to(DEV), "control": control, "transformer_options": {}}
    den = w(lambda *a, **k: (_ for _ in ()).throw(AssertionError("deferred")), {"input": x, "timestep": sigma, "c": c, "cond_or_uncond": [0]})
    torch.cuda.synchronize()
    assert w.calls_fast == 1
    xc = pred.calculate_input(sigma.cpu(), x.cpu())
    with torch.no_grad():
        eps = OU.unet_forward(sd, cfg, xc, pred.timestep(sigma.cpu()).float(), g["context"], g["y"], control=g["control"])
    assert_close("P3 wrapper + control vs oracle fp32", den, pred.calculate_denoised(sigma.cpu(), eps, x.cpu()), rel_rms=4e-3)


# ------------------------------------------------------------------------------------------------ f4: Chroma / RMSNorm
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("rows,C", [(300, 3072), (77, 5120), (1024, 64)])
def test_rmsnorm_rows(dtype, rows, C):
    from b200forge import ops
    x = _rand(rows, C, dtype=dtype, seed=4) * 2 + 0.3
    sc = (1 + 0.1 * _rand(C, dtype=torch.float32, seed=5)).to(dtype)
    y = ops.rmsnorm_rows(x, sc, 1e-6)
    torch.cuda.synchronize()
    xf = x.float()
    ref = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + 1e-6) * sc.float()
    assert_close(f"rmsnorm_rows {rows}x{C} {dtype}", y, ref, rel_rms=4e-3 if dtype == torch.bfloat16 else 6e-4)


def test_chroma_engine_vs_reference_golden():
    from b200forge.flux_engine import ChromaEngine
    from oracle import chroma as OC
    g = _gold("chroma_tiny.pt")
    cfg = OC.CONFIGS[g["config"]]
    sd = OC.random_state_dict(cfg, seed=g["weight_seed"])
    eng = ChromaEngine(cfg, sd, dtype=torch.bfloat16, device=DEV)
    out = eng.forward(g["x"].to(DEV), g["t"].to(DEV), g["context"].to(DEV).bfloat16())
    torch.cuda.synchronize()
    with torch.no_grad():  # the reference's own bf16 arithmetic on the same inputs (CPU: the oracle builds its index tables there)
        sd_bf = {k: v.bfloat16() for k, v in sd.items()}
        ref_bf = OC.chroma_forward(sd_bf, cfg, g["x"].bfloat16(), g["t"], g["context"].bfloat16()).float()
    r_ref = err_stats(ref_bf, g["out"])[1]
    m, r = err_stats(out, g["out"])
    print(f"[parity] chroma tiny bf16: ours rel_rms={r:.3e} max_abs={m:.3e}; oracle-in-bf16 rel_rms={r_ref:.3e}")
    assert torch.isfinite(out.float()).all() and r <= max(1.5 * r_ref, 3e-2)


# ------------------------------------------------------------------------------------------------ f2: LMS / SDE plans
@pytest.mark.parametrize("key", ["sample_lms", "sample_dpmpp_sde", "sample_dpmpp_2m_sde", "sample_dpmpp_2m_sde_heun", "sample_dpmpp_3m_sde",
                                 "sample_heunpp2", "sample_ipndm", "sample_ipndm_v", "sample_deis"])
def test_p4_lms_and_sde_samplers_vs_reference_golden(key):
    """Host plans of LMS (order 4), the three DPM++ SDE variants, Heun++ and the iPNDM / iPNDM-v / DEIS multistep samplers driving the update kernel on the device, against the
    reference's own k-diffusion loops around the same toy denoiser and noise stream (tests/golden/samplers_toy.pt)."""
    from b200forge import k_samplers
    g = _gold("samplers_toy.pt")
    name = key.replace("_heun", "") if key.endswith("sde_heun") else key
    kw = {"solver_type": "heun"} if key.endswith("sde_heun") else {}
    k = iter(range(g["noise"].shape[0]))
    if "sde" in name:
        kw["noise_sampler"] = lambda s, sn: g["noise"][next(k)].to(DEV)
    seen = []
    out = getattr(k_samplers, name)(lambda x, sigma, **kwargs: S.toy_denoiser(x, sigma), g["x0"].to(DEV), g["sigmas"].to(DEV),
                                    extra_args={}, callback=lambda d: seen.append(d["i"]), disable=True, **kw)
    torch.cuda.synchronize()
    assert seen == list(range(len(g["sigmas"]) - 1))
    assert_close(f"P4 {key} vs reference golden", out, g[key], rel_rms=3e-5)


def test_sampler_update_brings_foreign_noise_to_the_device():
    """ADVICE r1: noise / old_denoised are raw pointers for the kernel — a CPU tensor, a broadcast [1,C,H,W] draw or an fp64
    tensor from a user's noise_sampler must be brought to x's device / shape / dtype, not read out of bounds."""
    from b200forge import ops
    g = torch.Generator().manual_seed(6)
    x0 = torch.randn(3, 4, 8, 8, generator=g)
    den = torch.randn(3, 4, 8, 8, generator=g)
    n1 = torch.randn(1, 4, 8, 8, generator=g).double()  # CPU, fp64, batch-broadcast
    ref = x0 + ((x0 - den) / 2.0) * (-0.5) + n1.float() * 0.3
    x = x0.to(DEV).clone()
    ops.sampler_update(x, den.to(DEV), kind=ops.STEP_EULER, sigma=2.0, dt=-0.5, noise=n1, noise_scale=0.3)
    torch.cuda.synchronize()
    assert_close("sampler_update with a CPU fp64 broadcast noise", x, ref, max_abs=1e-5)
    with pytest.raises(RuntimeError):
        ops.sampler_update(x, den.to(DEV), kind=ops.STEP_EULER, sigma=2.0, dt=-0.5, noise=torch.randn(2, 4, 8, 8), noise_scale=0.3)


# ------------------------------------------------------------------------------------------------ v-prediction, hires-fix
def test_v_prediction_pipeline_vs_reference_trajectory():
    from b200forge.pipeline import Txt2ImgPipeline
    g = _gold("traj_tiny_21_v.pt")
    cfg = CF.CONFIGS[g["config"]]
    pipe = Txt2ImgPipeline(cfg, OU.random_state_dict(cfg, seed=g["weight_seed"]), dtype=torch.float16, device=DEV,
                           prediction_type="v_prediction")
    dens = []
    x = pipe.sample(g["cond"], g["uncond"], g["noise0"], sampler="euler", cfg_scale=g["cfg_scale"], sigmas=g["sigmas"],
                    callback=lambda i, xb, d: dens.append(d.clone()))
    torch.cuda.synchronize()
    assert_close("v-pred first denoised vs reference golden", dens[0], g["denoised0"], rel_rms=8e-3)
    mse = (x.cpu() - g["euler"]).pow(2).mean()
    psnr = float(10 * torch.log10(g["euler"].abs().max() ** 2 / mse))
    print(f"[parity] v-pred euler trajectory PSNR {psnr:.1f} dB")
    assert psnr >= 40.0, psnr


def test_hires_fix_vs_oracle_composition():
    """txt2img + latent hires-fix second pass (modules/processing.py:1342-1540, latent upscaler) on the device against the
    same composition of oracle pieces in fp32: Euler first pass, bilinear latent resize, Euler over the last t_enc+1 sigmas."""
    from b200forge.pipeline import Txt2ImgPipeline
    cfg = CF.CONFIGS["tiny_xl"]
    sd = OU.random_state_dict(cfg, seed=1)
    pipe = Txt2ImgPipeline(cfg, sd, dtype=torch.float16, device=DEV)
    g = torch.Generator().manual_seed(9)
    B, steps, strength = 2, 6, 0.5
    cond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g), vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    uncond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g), vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    noise = torch.randn(B, 4, 16, 16, generator=g)
    noise_hr = torch.randn(B, 4, 32, 32, generator=g)
    x = pipe.hires_fix(cond, uncond, noise, noise_hr, steps=steps, denoising_strength=strength, sampler="euler", cfg_scale=5.0)
    torch.cuda.synchronize()
    pred = S.EpsPrediction()
    s1 = S.get_sigmas_uniform(pred, steps)
    den = S.Denoiser(lambda xc, t, cx, yy: OU.unet_forward(sd, cfg, xc, t, cx, yy), pred, cond, uncond, 5.0)
    with torch.no_grad():
        first = S.sample_euler(den, noise * s1[0], s1)
        up = torch.nn.functional.interpolate(first, size=(32, 32), mode="bilinear", antialias=False)
        t_enc = int(min(strength, 0.999) * steps)
        sched = s1[steps - t_enc - 1:]
        ref = S.sample_euler(den, noise_hr * sched[0] + up, sched)
    mse = (x.cpu() - ref).pow(2).mean()
    psnr = float(10 * torch.log10(ref.abs().max() ** 2 / mse))
    print(f"[parity] hires-fix PSNR {psnr:.1f} dB")
    assert psnr >= 35.0, psnr


# ------------------------------------------------------------------------------------------------ non-square SDXL bucket
@pytest.mark.parametrize("route", ["generic", "im2col"])
def test_sdxl_full_width_non_square_bucket(route, monkeypatch):
    """SDXL 1216x832 (latent 152x104; levels 152x104, 76x52, 38x26 — none tiles into whole-row 128-pixel boxes) through the
    fused UNet at full width against the oracle in fp32, for both routes of the non-tiling convolutions; the attention
    runs over 3952 / 988 tokens (ragged query and key tiles).  Reference: backend/nn/unet.py:696-763 takes any H x W."""
    from b200forge import ops, synthetic
    from b200forge.unet_engine import UNetEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    monkeypatch.setenv("B200_CONV_ROUTE", route)
    cfg = synthetic.SDXL
    sd = synthetic.random_unet_state_dict(cfg, device=DEV, dtype=torch.float16, seed=0)
    eng = UNetEngine(cfg, sd, dtype=torch.float16, device=DEV)
    assert not ops.conv3x3_supported(104, 152) and eng.supports_latent(104, 152)
    g = torch.Generator().manual_seed(40)
    n = 2
    x = torch.randn(n, 4, 104, 152, generator=g).half().to(DEV)
    ctx = torch.randn(n, 77, 2048, generator=g).half().to(DEV)
    y = torch.randn(n, 2816, generator=g).half().to(DEV)
    t = torch.tensor([900.0, 50.0], device=DEV)
    out = eng.forward(x, t, ctx, y)
    torch.cuda.synchronize()
    with torch.no_grad():
        ref = OU.unet_forward({k: v.float() for k, v in sd.items()}, cfg, x.float(), t, ctx.float(), y.float())
    assert_close(f"SDXL 1216x832 ({route} route) fp16 engine vs oracle fp32", out, ref, rel_rms=3e-3)
    assert ((out.float() - ref).abs().max() / ref.pow(2).mean().sqrt()).item() <= 2e-2


def test_vae_decode_non_square_bucket():
    from b200forge import synthetic
    from b200forge.vae_engine import VAEDecoderEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = synthetic.VAE_SDXL
    sd = synthetic.random_vae_decoder_state_dict(cfg, device=DEV, dtype=torch.bfloat16, seed=1)
    eng = VAEDecoderEngine(cfg, sd, dtype=torch.bfloat16, device=DEV)
    assert eng.supports_latent(52, 76)
    g = torch.Generator().manual_seed(41)
    z = (torch.randn(1, 4, 52, 76, generator=g) * cfg["scaling_factor"]).to(DEV)
    img = eng.decode(z)
    torch.cuda.synchronize()
    with torch.no_grad():
        ref = OV.decode_first_stage({k: v.float() for k, v in sd.items()}, cfg, z)
        ref_bf = OV.decode_first_stage(sd, cfg, z.bfloat16()).float()
    r_ref = err_stats(ref_bf, ref)[1]
    m, r = err_stats(img, ref)
    print(f"[parity] vae 608x416: ours rel_rms={r:.3e} max_abs={m:.3e}; oracle-in-bf16 rel_rms={r_ref:.3e}")
    assert img.shape == (1, 416, 608, 3) and r <= max(1.5 * r_ref, 5e-3)


# ------------------------------------------------------------------------------------------------ GEMM alpha / scaled logits
def test_gemm_alpha_and_fp16_logit_range():
    """C = alpha * A B^T: the GEMM-softmax-GEMM attention paths store SCALED logits.  With Dh = 160 and |q|,|k| ~ 24 the
    unscaled fp16 logits overflow (160 * 24 * 24 = 92 160 > 65 504); the scaled ones (x 160^-1/2) do not."""
    from b200forge import ops
    a = _rand(256, 160, seed=7)
    w = _rand(512, 160, seed=8)
    y = ops.gemm(a, w, alpha=0.25)
    torch.cuda.synchronize()
    assert_close("gemm alpha", y, 0.25 * O.linear(a.float(), w.float()), max_abs=3e-2, rel_rms=1e-3)
    B, H, L, Dh = 2, 2, 64, 160
    q = torch.full((B, L, H * Dh), 24.0, dtype=torch.float16, device=DEV) + _rand(B, L, H * Dh, seed=9)
    k = torch.full((B, L, H * Dh), 24.0, dtype=torch.float16, device=DEV) + _rand(B, L, H * Dh, seed=10)
    v = _rand(B, L, H * Dh, seed=11)
    out = ops.attention_blockdiag(q, k, v, H, scale=Dh ** -0.5)
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()  # (logits this large are beyond fp16 resolution either way; the point is no inf / NaN)
    assert out.abs().max().item() <= v.abs().max().item() * 1.01  # a convex combination of the value rows


# ------------------------------------------------------------------------------------------------ f4: other LDM-UNet families
@pytest.mark.parametrize("name", ["sd21", "sdxl_refiner"])
def test_other_unet_families_full_width_vs_oracle_fp32(name):
    """SD2.x (4 levels, linear transformer, head dim 64, 1024-wide context, no label embedding) and the SDXL refiner (384 base
    channels, 4 transformer layers at levels 1-2, 1280-wide context, 2560-wide label embedding) are the same LDM UNet under
    other configurations: full width on a 32x32 latent against the oracle in fp32."""
    from b200forge import synthetic
    from b200forge.unet_engine import UNetEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = CF.CONFIGS[name]
    sd = synthetic.random_unet_state_dict(cfg, device=DEV, dtype=torch.float16, seed=3)
    eng = UNetEngine(cfg, sd, dtype=torch.float16, device=DEV)
    g = torch.Generator().manual_seed(60)
    n, hw = 2, 32
    x = torch.randn(n, 4, hw, hw, generator=g).half().to(DEV)
    ctx = torch.randn(n, 77, cfg["context_dim"], generator=g).half().to(DEV)
    y = torch.randn(n, cfg["adm_in_channels"], generator=g).half().to(DEV) if cfg["adm_in_channels"] else None
    t = torch.tensor([850.0, 120.0], device=DEV)
    out = eng.forward(x, t, ctx, y)
    torch.cuda.synchronize()
    with torch.no_grad():
        ref = OU.unet_forward({k: v.float() for k, v in sd.items()}, cfg, x.float(), t, ctx.float(), None if y is None else y.float())
    assert_close(f"unet {name} full width fp16 engine vs oracle fp32", out, ref, max_rel=2e-2, rel_rms=3e-3)
