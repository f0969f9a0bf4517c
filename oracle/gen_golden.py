"""ORACLE tooling — generates tests/golden/*.pt by running the UNMODIFIED reference (imported from
/root/reference through oracle/ref_import.py) on CPU fp32 with deterministic synthetic weights.

    python -m oracle.gen_golden            # in the build container (needs /root/reference)

The fixtures pin (a) the oracle restatement and (b) the CUDA path on the GPU box, where the reference tree
does not exist.  Weights are not stored: `oracle.unet.random_state_dict(cfg, seed)` regenerates them
bit-identically (CPU torch.Generator), and each fixture stores a checksum of the weights it was made with.
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import configs as CF  # noqa: E402
from oracle import ref_import  # noqa: E402
from oracle import unet as OU  # noqa: E402
from oracle.golden import GOLD, control_residuals, sample_index, seeded_inputs  # noqa: E402


def sd_checksum(sd) -> float:
    return float(sum(v.double().abs().sum() for v in sd.values()))


def make_inputs(cfg, B, hw, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 4, hw, hw, generator=g)
    ctx = torch.randn(B, 77, cfg["context_dim"], generator=g)
    y = torch.randn(B, cfg["adm_in_channels"], generator=g) if cfg.get("adm_in_channels") else None
    return x, ctx, y


def gen_unet(name: str, hw: int = 16):
    from backend.nn.unet import IntegratedUNet2DConditionModel as RefUNet
    cfg = CF.CONFIGS[name]
    sd = OU.random_state_dict(cfg, seed=1)
    m = RefUNet(**cfg).eval()
    m.load_state_dict(sd, strict=True)
    x, ctx, y = make_inputs(cfg, 2, hw, seed=2)
    t = torch.tensor([981.0, 23.0])
    with torch.no_grad():
        out = m(x, t, context=ctx, y=y, transformer_options={})
    torch.save(dict(config=name, weight_seed=1, weight_checksum=sd_checksum(sd), x=x, t=t, context=ctx, y=y, out=out),
               os.path.join(GOLD, f"unet_{name}.pt"))
    print("unet", name, "out std", out.std().item())


def gen_v_trajectory(name: str = "tiny_21", hw: int = 16, steps: int = 5):
    """SD2.x-style run: 4-level linear-transformer UNet without label_emb, v-prediction, Euler, CFG 6 — the reference's
    KModel.apply_model -> sampling_function_inner -> k_diffusion.sample_euler on CPU fp32."""
    import k_diffusion.sampling as ks
    from backend.modules.k_model import KModel
    from backend.modules.k_prediction import Prediction
    from backend.nn.unet import IntegratedUNet2DConditionModel as RefUNet
    from backend.sampling.condition import compile_conditions
    from backend.sampling.sampling_function import sampling_function_inner
    from k_diffusion.external import ForgeScheduleLinker
    ks.to_d = lambda x, sigma, denoised: (x - denoised) / sigma
    cfg = CF.CONFIGS[name]
    sd = OU.random_state_dict(cfg, seed=1)
    unet = RefUNet(**cfg).eval()
    unet.load_state_dict(sd, strict=True)
    unet.storage_dtype = torch.float32
    unet.computation_dtype = torch.float32
    pred = Prediction(prediction_type="v_prediction")
    kmodel = KModel(unet, diffusers_scheduler=None, k_predictor=pred)
    B = 2
    g = torch.Generator().manual_seed(17)
    cond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g))
    uncond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g))
    # SD1.x / 2.x conditioning is a bare tensor (condition.py:95-103): no pooled vector
    cond_c, uncond_c = compile_conditions(cond["crossattn"]), compile_conditions(uncond["crossattn"])
    cfg_scale = 6.0

    class Wrap:
        class _Inner:
            predictor = pred
        inner_model = _Inner()

        def __call__(self, x, sigma, **kw):
            return sampling_function_inner(kmodel, x, sigma, uncond_c, cond_c, cfg_scale, {}, None)

    sig = ForgeScheduleLinker(pred).get_sigmas(steps)
    noise0 = torch.randn(B, 4, hw, hw, generator=g)
    with torch.no_grad():
        # modules/sd_samplers_kdiffusion.py:207 with opts.sgm_noise_multiplier at its default False (shared_options.py:410)
        x0 = pred.noise_scaling(sig[0], noise0.clone(), torch.zeros_like(noise0), max_denoise=False)
        x = make_inputs(cfg, B, hw, seed=2)[0]
        fwd = unet(x, torch.tensor([981.0, 23.0]), context=cond["crossattn"], y=None, transformer_options={})
        dens = []
        out = ks.sample_euler(Wrap(), x0.clone(), sig, extra_args={}, callback=lambda d: dens.append(d["denoised"].clone()), disable=True)
    torch.save(dict(config=name, weight_seed=1, weight_checksum=sd_checksum(sd), cond=cond, uncond=uncond, cfg_scale=cfg_scale,
                    sigmas=sig, noise0=noise0, x0=x0, euler=out, denoised0=dens[0], fwd_x=x, fwd_t=torch.tensor([981.0, 23.0]),
                    fwd_out=fwd), os.path.join(GOLD, f"traj_{name}_v.pt"))
    print("v-pred traj", name, float(out.std()), float(fwd.std()))


def gen_trajectories(name: str = "tiny_xl", hw: int = 16, steps: int = 6):
    """Reference denoise loop: KModel.apply_model -> sampling_function_inner (CFG) -> k_diffusion sample_*."""
    import k_diffusion.sampling as ks
    from backend.modules.k_model import KModel
    from backend.modules.k_prediction import Prediction
    from backend.nn.unet import IntegratedUNet2DConditionModel as RefUNet
    from backend.sampling.condition import compile_conditions
    from backend.sampling.sampling_function import sampling_function_inner
    from k_diffusion.external import ForgeScheduleLinker

    # modules/sd_schedulers.py:10-15 replaces k_diffusion.sampling.to_d at import time; `modules` cannot be
    # imported here (gradio etc. missing), so the same override is applied by hand.
    ks.to_d = lambda x, sigma, denoised: (x - denoised) / sigma

    cfg = CF.CONFIGS[name]
    sd = OU.random_state_dict(cfg, seed=1)
    unet = RefUNet(**cfg).eval()
    unet.load_state_dict(sd, strict=True)
    unet.storage_dtype = torch.float32
    unet.computation_dtype = torch.float32
    pred = Prediction(prediction_type="epsilon")
    kmodel = KModel(unet, diffusers_scheduler=None, k_predictor=pred)
    linker = ForgeScheduleLinker(pred)

    B = 2
    g = torch.Generator().manual_seed(7)
    cond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g),
                vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    uncond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g),
                  vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    cond_c, uncond_c = compile_conditions(cond), compile_conditions(uncond)
    cfg_scale = 7.0

    class Wrap:  # what k-diffusion sees as `model`: CFGDenoiser minus UI glue (sd_samplers_cfg_denoiser.py:199)
        class _Inner:
            predictor = pred
        inner_model = _Inner()

        def __call__(self, x, sigma, **kw):
            return sampling_function_inner(kmodel, x, sigma, uncond_c, cond_c, cfg_scale, {}, None)

    seeds = [1000, 1001]
    gens = [torch.Generator().manual_seed(s) for s in seeds]

    def draw():  # modules/rng.py:167-177 ImageRNG.next(): one randn per image generator, stacked
        return torch.stack([torch.randn((4, hw, hw), generator=gg) for gg in gens])

    sig_auto = linker.get_sigmas(steps)                       # Euler / Euler a "Automatic" schedule
    sig_karras = ks.get_sigmas_karras(steps, float(pred.sigma_min), float(pred.sigma_max))
    out = dict(config=name, weight_seed=1, weight_checksum=sd_checksum(sd), cond=cond, uncond=uncond,
               cfg_scale=cfg_scale, seeds=seeds, hw=hw, steps=steps, sigmas_auto=sig_auto, sigmas_karras=sig_karras)
    with torch.no_grad():
        noise0 = draw()
        # modules/sd_samplers_kdiffusion.py:207: max_denoise = opts.sgm_noise_multiplier, default False (shared_options.py:410)
        x0 = pred.noise_scaling(sig_auto[0], noise0.clone(), torch.zeros_like(noise0), max_denoise=False)
        out["noise0"] = noise0
        out["x0"] = x0
        step_noise = []

        class Hijack:  # TorchHijack (modules/sd_samplers_common.py:214-235): randn_like -> ImageRNG.next
            @staticmethod
            def randn_like(x):
                n = draw()
                step_noise.append(n)
                return n

            def __getattr__(self, item):
                return getattr(torch, item)

        ks.torch = Hijack()
        try:
            dens = []
            cb = lambda d: dens.append(d["denoised"].clone())  # noqa: E731
            out["euler_a"] = ks.sample_euler_ancestral(Wrap(), x0.clone(), sig_auto, extra_args={}, callback=cb, disable=True)
            out["euler_a_step_noise"] = torch.stack(step_noise)
            out["euler_a_denoised0"] = dens[0]
            out["euler_a_denoised_last"] = dens[-1]
            step_noise.clear()
            out["euler"] = ks.sample_euler(Wrap(), x0.clone(), sig_auto, extra_args={}, disable=True)
            x0k = pred.noise_scaling(sig_karras[0], noise0.clone(), torch.zeros_like(noise0), max_denoise=False)
            out["x0_karras"] = x0k
            out["dpmpp_2m"] = ks.sample_dpmpp_2m(Wrap(), x0k.clone(), sig_karras, extra_args={}, disable=True)
            # one run with the "SGM noise multiplier" option on (max_denoise=True)
            x0s = pred.noise_scaling(sig_auto[0], noise0.clone(), torch.zeros_like(noise0), max_denoise=True)
            out["x0_sgm"] = x0s
            out["euler_sgm"] = ks.sample_euler(Wrap(), x0s.clone(), sig_auto, extra_args={}, disable=True)
        finally:
            ks.torch = torch
    torch.save(out, os.path.join(GOLD, f"traj_{name}.pt"))
    print("traj", name, {k: float(v.std()) for k, v in out.items() if k in ("euler_a", "euler", "dpmpp_2m")})


def gen_schedules():
    import k_diffusion.sampling as ks
    from backend.modules.k_prediction import Prediction
    from k_diffusion.external import ForgeScheduleLinker
    pred = Prediction(prediction_type="epsilon")
    linker = ForgeScheduleLinker(pred)
    probe = torch.tensor([14.6146, 10.0, 3.3, 1.0, 0.5, 0.1, 0.0292])
    out = dict(sigmas=pred.sigmas.clone(), auto20=linker.get_sigmas(20), auto30=linker.get_sigmas(30),
               karras30=ks.get_sigmas_karras(30, float(pred.sigma_min), float(pred.sigma_max)),
               probe=probe, probe_timestep=pred.timestep(probe))
    torch.save(out, os.path.join(GOLD, "schedules.pt"))
    print("schedules sigma_min/max", float(pred.sigma_min), float(pred.sigma_max))


def gen_vae(name: str = "tiny", hw: int = 16):
    from backend.nn.vae import IntegratedAutoencoderKL
    from oracle import vae as OV
    cfg = CF.VAE_CONFIGS[name]
    sd = OV.random_state_dict(cfg, seed=3)
    m = IntegratedAutoencoderKL(**{k: v for k, v in cfg.items()}).eval()
    missing = m.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys, missing
    assert all(k.startswith(("encoder.", "quant_conv.")) for k in missing.missing_keys), missing.missing_keys
    g = torch.Generator().manual_seed(4)
    z = torch.randn(2, cfg["latent_channels"], hw, hw, generator=g)
    with torch.no_grad():
        out = m.decode(m.process_out(z))
    torch.save(dict(config=name, weight_seed=3, weight_checksum=sd_checksum(sd), z=z, out=out),
               os.path.join(GOLD, f"vae_{name}.pt"))
    print("vae", name, "out std", out.std().item())


def gen_vae_tiled(name: str = "tiny"):
    """The reference's tiled decode: its own `tiled_scale` (backend/patcher/vae.py:11-57) around its own
    IntegratedAutoencoderKL.decode, composed as VAE.decode_tiled_ composes them (:104-115; the VAE wrapper class itself needs
    the memory manager and a loaded model, the three-line composition is restated here)."""
    from backend.nn.vae import IntegratedAutoencoderKL
    from backend.patcher.vae import tiled_scale
    from oracle import vae as OV
    cfg = CF.VAE_CONFIGS[name]
    sd = OV.random_state_dict(cfg, seed=3)
    m = IntegratedAutoencoderKL(**{k: v for k, v in cfg.items()}).eval()
    m.load_state_dict(sd, strict=False)
    g = torch.Generator().manual_seed(6)
    z = torch.randn(2, cfg["latent_channels"], 20, 28, generator=g)
    tile_x = tile_y = 8
    overlap = 2
    up = 2 ** (len(cfg["block_out_channels"]) - 1)
    fn = lambda a: (m.decode(a) + 1.0).float()  # noqa: E731
    with torch.no_grad():
        zz = m.process_out(z)
        out = torch.clamp(((tiled_scale(zz, fn, tile_x // 2, tile_y * 2, overlap, upscale_amount=up) +
                            tiled_scale(zz, fn, tile_x * 2, tile_y // 2, overlap, upscale_amount=up) +
                            tiled_scale(zz, fn, tile_x, tile_y, overlap, upscale_amount=up)) / 3.0) / 2.0, min=0.0, max=1.0)
    torch.save(dict(config=name, weight_seed=3, weight_checksum=sd_checksum(sd), z=z, tile_x=tile_x, tile_y=tile_y, overlap=overlap,
                    out=out.movedim(1, -1)), os.path.join(GOLD, f"vae_tiled_{name}.pt"))
    print("vae tiled", name, "out std", out.std().item(), tuple(out.shape))


def gen_samplers(steps: int = 7):
    """The reference's own k-diffusion loops (k_diffusion/sampling.py) on CPU fp32 around oracle.sampling.toy_denoiser,
    with the to_d override of modules/sd_schedulers.py:10-15 and a recorded noise stream."""
    import k_diffusion.sampling as ks
    from backend.modules.k_prediction import Prediction
    from oracle import sampling as OS
    ks.to_d = lambda x, sigma, denoised: (x - denoised) / sigma
    pred = Prediction(prediction_type="epsilon")
    sig = ks.get_sigmas_karras(steps, float(pred.sigma_min), float(pred.sigma_max))
    g = torch.Generator().manual_seed(11)
    x0 = torch.randn(2, 4, 16, 16, generator=g) * sig[0]
    noise = torch.randn(4 * steps, 2, 4, 16, 16, generator=g)

    class Model:
        class _Inner:
            predictor = pred
        inner_model = _Inner()

        def __call__(self, x, sigma, **kw):
            return OS.toy_denoiser(x, sigma)

    out = dict(sigmas=sig, x0=x0, noise=noise)
    runs = [("sample_heun", {}), ("sample_dpm_2", {}), ("sample_dpm_2_ancestral", {}), ("sample_dpmpp_2s_ancestral", {}),
            ("sample_lms", {}), ("sample_dpmpp_sde", {}), ("sample_dpmpp_2m_sde", {}),
            ("sample_dpmpp_2m_sde", {"solver_type": "heun"}), ("sample_dpmpp_3m_sde", {}),
            ("sample_heunpp2", {}), ("sample_ipndm", {}), ("sample_ipndm_v", {}), ("sample_deis", {})]
    for name, extra in runs:
        k = iter(range(noise.shape[0]))
        kw = dict(extra)
        if "ancestral" in name or "sde" in name:
            kw["noise_sampler"] = lambda s, sn: noise[next(k)]
        key = name + ("_heun" if extra.get("solver_type") == "heun" else "")
        with torch.no_grad():
            out[key] = getattr(ks, name)(Model(), x0.clone(), sig, extra_args={}, disable=True, **kw)
        print(key, float(out[key].std()))
    # Restart (modules/sd_samplers_extra.py imports only torch / tqdm / k_diffusion, so the reference file itself is run):
    # 24 steps so that the automatic restart list is non-empty (steps >= 20); noise through k_diffusion.sampling.torch
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_sd_samplers_extra", os.path.join(ref_import.REF_ROOT, "modules", "sd_samplers_extra.py"))
    extra = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(extra)
    sig24 = ks.get_sigmas_karras(24, float(pred.sigma_min), float(pred.sigma_max))
    x24 = torch.randn(2, 4, 16, 16, generator=torch.Generator().manual_seed(13)) * sig24[0]
    rn = torch.randn(8, 2, 4, 16, 16, generator=torch.Generator().manual_seed(14))
    kk = iter(range(8))

    class Hijack:
        @staticmethod
        def randn_like(x):
            return rn[next(kk)]

        def __getattr__(self, item):
            return getattr(torch, item)

    ks.torch = Hijack()
    try:
        with torch.no_grad():
            out["restart_sampler"] = extra.restart_sampler(Model(), x24.clone(), sig24, extra_args={}, disable=True)
    finally:
        ks.torch = torch
    out["restart_sigmas"], out["restart_x0"], out["restart_noise"] = sig24, x24, rn
    print("restart_sampler", float(out["restart_sampler"].std()), "noise draws used", next(kk))
    # rectified-flow variants: the reference dispatches on isinstance(model.inner_model.predictor, PredictionFlux)
    from backend.modules.k_prediction import PredictionFlux
    from oracle import sampling as OS2
    fpred = PredictionFlux()
    fsig = OS2.simple_scheduler(steps, OS2.flux_sigma_table())

    class FluxModel(Model):
        class _Inner:
            predictor = fpred
        inner_model = _Inner()

    xf0 = torch.randn(2, 4, 16, 16, generator=torch.Generator().manual_seed(12)) * fsig[0]
    out["flux_sigmas"], out["flux_x0"] = fsig, xf0
    for name in ("sample_euler_ancestral", "sample_dpm_2_ancestral"):
        k = iter(range(noise.shape[0]))
        with torch.no_grad():
            out[name + "_rf"] = getattr(ks, name)(FluxModel(), xf0.clone(), fsig, extra_args={}, disable=True,
                                                  noise_sampler=lambda s, sn: noise[next(k)])
        print(name + "_rf", float(out[name + "_rf"].std()))
    torch.save(out, os.path.join(GOLD, "samplers_toy.pt"))


def gen_vae_encode(name: str = "tiny", hw: int = 64):
    """Reference IntegratedAutoencoderKL.encode (backend/nn/vae.py:293-303): moments via a `regulation` hook, and the
    default .sample() with the global CPU generator seeded (the reference draws torch.randn(mean.shape) there)."""
    from backend.nn.vae import IntegratedAutoencoderKL
    from oracle import vae as OV
    cfg = CF.VAE_CONFIGS[name]
    sd = OV.random_encoder_state_dict(cfg, seed=8)
    m = IntegratedAutoencoderKL(**{k: v for k, v in cfg.items()}).eval()
    missing = m.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys, missing
    assert all(k.startswith(("decoder.", "post_quant_conv.")) for k in missing.missing_keys), missing.missing_keys
    g = torch.Generator().manual_seed(9)
    pixels = torch.rand(2, hw, hw, 3, generator=g)                       # NHWC in [0, 1], what VAE.encode receives
    x = 2.0 * pixels.movedim(-1, 1) - 1.0                                # patcher/vae.py:177
    with torch.no_grad():
        mean, logvar = m.encode(x, regulation=lambda p: (p.mean, p.logvar))
        torch.manual_seed(1234)
        sample = m.encode(x)
        torch.manual_seed(1234)
        noise = torch.randn(mean.shape)
    latent = m.process_in(sample)
    torch.save(dict(config=name, weight_seed=8, weight_checksum=sd_checksum(sd), pixels=pixels, mean=mean, logvar=logvar,
                    noise=noise, sample=sample, latent=latent), os.path.join(GOLD, f"vae_enc_{name}.pt"))
    print("vae encode", name, "mean std", mean.std().item(), "logvar mean", logvar.mean().item())


def gen_unet_control(name: str = "tiny_xl", hw: int = 16):
    """Reference UNet forward with ControlNet-style residuals (backend/nn/unet.py:44-52, 714, 733, 739): one tensor per input
    block, one for the middle block, one per output skip, plus a None entry, consumed from the end of each list."""
    from backend.nn.unet import IntegratedUNet2DConditionModel as RefUNet
    cfg = CF.CONFIGS[name]
    sd = OU.random_state_dict(cfg, seed=1)
    m = RefUNet(**cfg).eval()
    m.load_state_dict(sd, strict=True)
    x, ctx, y = make_inputs(cfg, 2, hw, seed=2)
    t = torch.tensor([981.0, 23.0])
    # shapes of the activations the residuals are added to: run once with hooks
    shapes = {"input": [], "middle": [], "output": []}
    hooks = [blk.register_forward_hook(lambda mod, i, o, k="input": shapes[k].append(tuple(o.shape))) for blk in m.input_blocks]
    hooks.append(m.middle_block.register_forward_hook(lambda mod, i, o: shapes["middle"].append(tuple(o.shape))))
    with torch.no_grad():
        m(x, t, context=ctx, y=y, transformer_options={})
    for h in hooks:
        h.remove()
    control_shapes = {"input": shapes["input"], "middle": shapes["middle"][:1]}
    control = control_residuals(control_shapes, seed=19)
    with torch.no_grad():
        out = m(x, t, context=ctx, y=y, control={k: list(v) for k, v in control.items()}, transformer_options={})
    # the residuals are not stored: control_residuals() regenerates them from the seed and shapes
    torch.save(dict(config=name, weight_seed=1, weight_checksum=sd_checksum(sd), x=x, t=t, context=ctx, y=y,
                    control_seed=19, control_shapes=control_shapes, out=out), os.path.join(GOLD, f"unet_{name}_control.pt"))
    print("unet control", name, "out std", out.std().item())


def gen_chroma(name: str = "tiny_chroma", hw: int = 16, txt_len: int = 64):
    """Reference Chroma transformer (backend/nn/chroma.py) on CPU fp32."""
    from backend.nn.chroma import IntegratedChromaTransformer2DModel
    from oracle import chroma as OC
    cfg = OC.CONFIGS[name]
    sd = OC.random_state_dict(cfg, seed=5)
    m = IntegratedChromaTransformer2DModel(**cfg).eval()
    m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(6)
    x = torch.randn(2, cfg["in_channels"], hw, hw_w or hw, generator=g)
    ctx = torch.randn(2, txt_len, cfg["context_in_dim"], generator=g)
    t = torch.tensor([0.93, 0.12])
    with torch.no_grad():
        out = m(x, t, ctx)
    torch.save(dict(config=name, weight_seed=5, weight_checksum=sd_checksum(sd), x=x, t=t, context=ctx, out=out),
               os.path.join(GOLD, "chroma_tiny.pt"))
    print("chroma", name, "out std", out.std().item())


def gen_flux(name: str = "tiny_flux", hw: int = 16, txt_len: int = 128, fname: str = "flux_tiny.pt", hw_w: int = None):
    """Reference Flux transformer (backend/nn/flux.py) on CPU fp32, distilled-guidance input included."""
    from backend.nn.flux import IntegratedFluxTransformer2DModel
    from oracle import flux as OF
    cfg = OF.CONFIGS[name]
    sd = OF.random_state_dict(cfg, seed=5)
    m = IntegratedFluxTransformer2DModel(**cfg).eval()
    m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(6)
    x = torch.randn(2, cfg["in_channels"], hw, hw_w or hw, generator=g)
    ctx = torch.randn(2, txt_len, cfg["context_in_dim"], generator=g)
    y = torch.randn(2, cfg["vec_in_dim"], generator=g)
    t = torch.tensor([0.93, 0.12])
    guidance = torch.tensor([4.0, 4.0])  # 4000 is exact in bf16 (3.5 * 1000 rounds to 3504 in the reference's bf16 run)
    with torch.no_grad():
        out = m(x, t, ctx, y, guidance)
    torch.save(dict(config=name, weight_seed=5, weight_checksum=sd_checksum(sd), x=x, t=t, context=ctx, y=y,
                    guidance=guidance, out=out), os.path.join(GOLD, fname))
    print("flux", name, "out std", out.std().item())


def gen_unet_b1(name: str = "tiny_xl"):
    """A second reference UNet forward at other weights / shape / timestep: batch 1, 8 x 8 latent, t = 400."""
    from backend.nn.unet import IntegratedUNet2DConditionModel as RefUNet
    cfg = CF.CONFIGS[name]
    sd = OU.random_state_dict(cfg, seed=5)
    m = RefUNet(**cfg).eval()
    m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(6)
    x = torch.randn(1, 4, 8, 8, generator=g)
    ctx = torch.randn(1, 77, cfg["context_dim"], generator=g)
    y = torch.randn(1, cfg["adm_in_channels"], generator=g)
    t = torch.tensor([400.0])
    with torch.no_grad():
        out = m(x, t, context=ctx, y=y, transformer_options={})
    torch.save(dict(config=name, weight_seed=5, weight_checksum=sd_checksum(sd), x=x, t=t, context=ctx, y=y, out=out),
               os.path.join(GOLD, f"unet_{name}_b1.pt"))
    print("unet b1", name, "out std", out.std().item())


def gen_param_shapes():
    """Parameter names and shapes of the reference's full-size SD1.5 / SDXL UNets and Flux.1-dev transformer (built on
    the meta device), stored as gzipped JSON {model: {name: shape}}."""
    import gzip
    import json

    from backend.nn.flux import IntegratedFluxTransformer2DModel
    from backend.nn.unet import IntegratedUNet2DConditionModel as RefUNet
    from oracle import flux as OF
    out = {}
    for key, ctor in (("sd15", lambda: RefUNet(**CF.CONFIGS["sd15"])), ("sdxl", lambda: RefUNet(**CF.CONFIGS["sdxl"])),
                      ("flux_dev", lambda: IntegratedFluxTransformer2DModel(**OF.FLUX_DEV))):
        with torch.device("meta"):
            m = ctor()
        out[key] = {k: list(p.shape) for k, p in m.named_parameters()}
        print("param shapes", key, len(out[key]), sum(p.numel() for p in m.parameters()))
    with gzip.GzipFile(os.path.join(GOLD, "param_shapes.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(out, separators=(",", ":"), sort_keys=True).encode())


def _detach(obj):
    """Tensors cloned, containers walked, anything else dropped (callables, model handles in transformer_options)."""
    if torch.is_tensor(obj):
        return obj.detach().clone()
    if isinstance(obj, dict):
        return {k: _detach(v) for k, v in obj.items() if torch.is_tensor(v) or isinstance(v, (dict, list, tuple, int, float, str, bool, type(None)))}
    if isinstance(obj, (list, tuple)):
        return type(obj)(_detach(v) for v in obj)
    return obj


def _record_wrapper_call(kmodel, x, sigma, uc, cc, cfg_scale):
    """Run the reference's sampling_function_inner with a model_function_wrapper that records what it is handed and what
    the reference's own apply_model returns for it."""
    from backend.sampling.sampling_function import sampling_function_inner
    calls = []

    def rec(apply_model, args):
        out = apply_model(args["input"], args["timestep"], **args["c"])
        calls.append(dict(args=_detach(args), out=out.detach().clone(), timestep_from_sigma=kmodel.predictor.timestep(args["timestep"]).clone()))
        return out

    with torch.no_grad():
        base = sampling_function_inner(kmodel, x, sigma, uc, cc, cfg_scale, {}, None)
        got = sampling_function_inner(kmodel, x, sigma, uc, cc, cfg_scale, {"model_function_wrapper": rec}, None)
    assert torch.equal(base, got) and len(calls) == 1, len(calls)
    return dict(calls[0], prediction_type=kmodel.predictor.prediction_type)


def gen_plugin_calls():
    """What the reference hands the plug points, and what its own code returns for it:
    - P1: the modules that import attention_function by value, and the attention_pytorch result on one input; the
      signature (shapes, heads, layout arguments) of each distinct attention call made by the reference UNet (tiny_xl) and
      Flux transformer (tiny) forwards of unet_tiny_xl.pt / flux_tiny.pt, with a sample of the reference's result on
      seeded inputs of those shapes;
    - P3: the model_function_wrapper call made by sampling_function_inner for a tiny_xl UNet (CFG 7) and a tiny Flux
      transformer (CFG 1), with the result of the reference's apply_model for the same arguments."""
    import backend.attention as ba
    import backend.nn.chroma  # noqa: F401
    import backend.nn.flux as bf
    import backend.nn.unet as bu
    import backend.nn.vae  # noqa: F401
    from backend.modules.k_model import KModel
    from backend.modules.k_prediction import Prediction, PredictionFlux
    from backend.sampling.condition import compile_conditions
    from oracle import flux as OF
    out = {}
    out["attention_importers"] = sorted(n for n, m in list(sys.modules.items())
                                        if m is not None and n != "backend.attention" and getattr(m, "attention_function", None) is ba.attention_function)
    out["single_head_importers"] = sorted(n for n, m in list(sys.modules.items()) if m is not None and n != "backend.attention"
                                          and getattr(m, "attention_function_single_head_spatial", None) is ba.attention_function_single_head_spatial)
    out["attention_function_name"] = ba.attention_function.__name__
    q = torch.randn(2, 16, 128, generator=torch.Generator().manual_seed(15))
    out["deferred_q"], out["deferred_out"] = q, ba.attention_function(q, q, q, 2)

    def record_attention(mod, model, inputs):
        """The first call of each distinct signature; replayed on seeded inputs of the same shapes (what is stored is the
        seed and a seeded sample of the reference's output)."""
        seen, calls = set(), []
        orig = mod.attention_function

        def rec(q, k, v, heads, *a, **kw):
            sig = (tuple(q.shape), tuple(k.shape), tuple(v.shape), heads, a, tuple(sorted(kw.items())))
            if sig not in seen:
                seen.add(sig)
                calls.append(sig)
            return orig(q, k, v, heads, *a, **kw)
        mod.attention_function = rec
        try:
            with torch.no_grad():
                model(*inputs[0], **inputs[1])
        finally:
            mod.attention_function = orig
        out = []
        for i, (qs, ks, vs, heads, a, kw) in enumerate(calls):
            seed = 100 + i
            q, k, v = seeded_inputs((qs, ks, vs), seed)
            with torch.no_grad():
                o = orig(q, k, v, heads, *a, **dict(kw))
            idx = sample_index(o.numel(), seed)
            out.append(dict(shapes=(qs, ks, vs), heads=heads, args=a, kwargs=dict(kw), seed=seed, out_shape=tuple(o.shape),
                            out_sample=o.reshape(-1)[idx].clone()))
        return out

    g = torch.load(os.path.join(GOLD, "unet_tiny_xl.pt"), weights_only=False)
    cfg = CF.CONFIGS["tiny_xl"]
    m = bu.IntegratedUNet2DConditionModel(**cfg).eval()
    m.load_state_dict(OU.random_state_dict(cfg, seed=g["weight_seed"]), strict=True)
    out["unet_attention_calls"] = record_attention(bu, m, ((g["x"], g["t"]), dict(context=g["context"], y=g["y"], transformer_options={})))
    gf = torch.load(os.path.join(GOLD, "flux_tiny.pt"), weights_only=False)
    fcfg = OF.CONFIGS[gf["config"]]
    fm = bf.IntegratedFluxTransformer2DModel(**fcfg).eval()
    fm.load_state_dict(OF.random_state_dict(fcfg, seed=gf["weight_seed"]), strict=True)
    out["flux_attention_calls"] = record_attention(bf, fm, ((gf["x"], gf["t"], gf["context"], gf["y"], gf["guidance"]), {}))
    print("attention calls recorded", len(out["unet_attention_calls"]), len(out["flux_attention_calls"]), out["attention_importers"])

    # P3, UNet
    sd = OU.random_state_dict(cfg, seed=1)
    unet = bu.IntegratedUNet2DConditionModel(**cfg).eval()
    unet.load_state_dict(sd, strict=True)
    unet.storage_dtype = unet.computation_dtype = torch.float32
    kmodel = KModel(unet, diffusers_scheduler=None, k_predictor=Prediction(prediction_type="epsilon"))
    g = torch.Generator().manual_seed(3)
    B = 2
    cond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g), vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    uncond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g), vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    x = torch.randn(B, 4, 16, 16, generator=g) * 4
    out["p3_unet"] = dict(config="tiny_xl", weight_seed=1,
                          **_record_wrapper_call(kmodel, x, torch.tensor([6.0, 6.0]), compile_conditions(uncond), compile_conditions(cond), 7.0))
    # P3, Flux
    fcfg = OF.TINY_FLUX
    fsd = OF.random_state_dict(fcfg, seed=5)
    fm = bf.IntegratedFluxTransformer2DModel(**fcfg).eval()
    fm.load_state_dict(fsd, strict=True)
    fm.storage_dtype = fm.computation_dtype = torch.float32
    kmodel = KModel(fm, diffusers_scheduler=None, k_predictor=PredictionFlux())
    g = torch.Generator().manual_seed(6)
    cond = dict(crossattn=torch.randn(B, 64, fcfg["context_in_dim"], generator=g), vector=torch.randn(B, fcfg["vec_in_dim"], generator=g),
                guidance=torch.full((B,), 4.0))
    x = torch.randn(B, 16, 16, 16, generator=g)
    out["p3_flux"] = dict(config="tiny_flux", weight_seed=5,
                          **_record_wrapper_call(kmodel, x, torch.tensor([0.8, 0.8]), None, compile_conditions(cond), 1.0))
    for k in ("p3_unet", "p3_flux"):
        print(k, {a: (tuple(v.shape) if torch.is_tensor(v) else v) for a, v in out[k]["args"]["c"].items()})
    torch.save(out, os.path.join(GOLD, "plugin_calls.pt"))


def gen_module_calls():
    """P2: every Linear / Conv2d / GroupNorm / LayerNorm module the reference UNet (tiny_xl), VAE decoder (tiny) and Flux
    transformer (tiny) run in the forwards of unet_tiny_xl.pt / vae_tiny.pt / flux_tiny.pt — its constructor arguments,
    state-dict name and input shape; the first module of each distinct (constructor, input shape) is run once more on a
    seeded input of that shape and a seeded sample of its output is stored."""
    from backend.nn.flux import IntegratedFluxTransformer2DModel
    from backend.nn.unet import IntegratedUNet2DConditionModel as RefUNet
    from backend.nn.vae import IntegratedAutoencoderKL
    from oracle import flux as OF
    from oracle import vae as OV
    nn = torch.nn

    def ctor(mod):
        if isinstance(mod, nn.Linear):
            return "Linear", dict(in_features=mod.in_features, out_features=mod.out_features, bias=mod.bias is not None)
        if isinstance(mod, nn.Conv2d):
            return "Conv2d", dict(in_channels=mod.in_channels, out_channels=mod.out_channels, kernel_size=mod.kernel_size,
                                  stride=mod.stride, padding=mod.padding, bias=mod.bias is not None)
        if isinstance(mod, nn.GroupNorm):
            return "GroupNorm", dict(num_groups=mod.num_groups, num_channels=mod.num_channels, eps=mod.eps, affine=mod.affine)
        if isinstance(mod, nn.LayerNorm):
            return "LayerNorm", dict(normalized_shape=tuple(mod.normalized_shape), eps=mod.eps, elementwise_affine=mod.elementwise_affine)
        return None

    def record(model, run):
        calls, seen, hooks = [], set(), []
        for name, mod in model.named_modules():
            c = ctor(mod)
            if c is None:
                continue

            def hook(m, inp, o, name=name, c=c):
                sig = (c[0], tuple(sorted(c[1].items())), tuple(inp[0].shape))
                entry = dict(name=name, kind=c[0], kwargs=c[1], x_shape=tuple(inp[0].shape))
                if sig not in seen:
                    seen.add(sig)
                    entry["replay"] = m
                calls.append(entry)
            hooks.append(mod.register_forward_hook(hook))
        try:
            with torch.no_grad():
                run()
        finally:
            for h in hooks:
                h.remove()
        for i, entry in enumerate(c for c in calls if "replay" in c):
            mod = entry.pop("replay")
            seed = 200 + i
            x, = seeded_inputs((entry["x_shape"],), seed)
            with torch.no_grad():
                o = mod(x)
            idx = sample_index(o.numel(), seed)
            entry.update(seed=seed, out_shape=tuple(o.shape), out_sample=o.reshape(-1)[idx].clone())
        return calls

    out = {}
    g = torch.load(os.path.join(GOLD, "unet_tiny_xl.pt"), weights_only=False)
    cfg = CF.CONFIGS[g["config"]]
    m = RefUNet(**cfg).eval()
    m.load_state_dict(OU.random_state_dict(cfg, seed=g["weight_seed"]), strict=True)
    out["unet"] = dict(config=g["config"], weight_seed=g["weight_seed"],
                       calls=record(m, lambda: m(g["x"], g["t"], context=g["context"], y=g["y"], transformer_options={})))
    gv = torch.load(os.path.join(GOLD, "vae_tiny.pt"), weights_only=False)
    vcfg = CF.VAE_CONFIGS[gv["config"]]
    vae = IntegratedAutoencoderKL(**vcfg).eval()
    vae.load_state_dict(OV.random_state_dict(vcfg, seed=gv["weight_seed"]), strict=False)
    out["vae"] = dict(config=gv["config"], weight_seed=gv["weight_seed"], calls=record(vae, lambda: vae.decode(vae.process_out(gv["z"]))))
    gf = torch.load(os.path.join(GOLD, "flux_tiny.pt"), weights_only=False)
    fcfg = OF.CONFIGS[gf["config"]]
    fm = IntegratedFluxTransformer2DModel(**fcfg).eval()
    fm.load_state_dict(OF.random_state_dict(fcfg, seed=gf["weight_seed"]), strict=True)
    out["flux"] = dict(config=gf["config"], weight_seed=gf["weight_seed"],
                       calls=record(fm, lambda: fm(gf["x"], gf["t"], gf["context"], gf["y"], gf["guidance"])))
    for k, v in out.items():
        kinds = {}
        for c in v["calls"]:
            kinds[c["kind"]] = kinds.get(c["kind"], 0) + 1
        print("module calls", k, kinds, "replayed:", sum(1 for c in v["calls"] if "seed" in c))
    torch.save(out, os.path.join(GOLD, "module_calls.pt"))


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    ref_import.load()
    which = sys.argv[1:] or ["unet", "traj", "vtraj", "sched", "samplers", "vae", "vae_tiled", "vae_enc", "control", "chroma", "flux", "flux_odd",
                             "unet_b1", "param_shapes", "plugin_calls", "module_calls"]
    if "unet" in which:
        gen_unet("tiny_xl")
        gen_unet("tiny_15")
        gen_unet("tiny_15h")
    if "traj" in which:
        gen_trajectories("tiny_xl")
    if "vtraj" in which:
        gen_v_trajectory("tiny_21")
    if "sched" in which:
        gen_schedules()
    if "vae" in which:
        gen_vae("tiny")
    if "vae_tiled" in which:
        gen_vae_tiled("tiny")
    if "samplers" in which:
        gen_samplers()
    if "vae_enc" in which:
        gen_vae_encode("tiny")
    if "control" in which:
        gen_unet_control("tiny_xl")
    if "chroma" in which:
        gen_chroma()
    if "flux" in which:
        gen_flux()                                                  # 64 img + 128 txt tokens: per-stream GEMM launches
        gen_flux(hw=32, txt_len=256, fname="flux_tiny_seg.pt")      # 256 + 256 tokens: two-segment GEMM path
    if "flux_odd" in which:
        gen_flux(hw=15, hw_w=18, txt_len=64, fname="flux_tiny_odd.pt")  # odd height: circular pad to the patch size + crop
    if "unet_b1" in which:
        gen_unet_b1()
    if "param_shapes" in which:
        gen_param_shapes()
    if "plugin_calls" in which:
        gen_plugin_calls()
    if "module_calls" in which:
        gen_module_calls()
