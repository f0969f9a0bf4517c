"""Host logic of the engines, pipelines and weight packing, pinned on the CPU: every `b200forge.ops` kernel wrapper is
replaced by its torch emulation (tests/ops_emulator.py) and the engines run in fp32, so their output must match the
reference goldens (tests/golden, made by the imported reference) to ~1e-4 — far tighter than the fp16/bf16 tolerances of the
GPU parity tests, which is what exposes packing / folding / ordering mistakes.  The CUDA kernels themselves are NOT
exercised here (that is what `-m gpu` does through the C ABI)."""
import sys
import types

import pytest
import torch

from oracle import configs as CF
from oracle import flux as OF
from oracle import sampling as S
from oracle import unet as OU
from oracle import vae as OV
from oracle.golden import load_golden, sample_index, seeded_inputs
from tests import ops_emulator
from tests.util import assert_close

F32 = torch.float32


def _gold(name):
    return load_golden(name)


@pytest.fixture(autouse=True)
def _emulated_ops(monkeypatch):
    ops_emulator.install(monkeypatch)


@pytest.mark.parametrize("name", ["tiny_xl", "tiny_15", "tiny_15h"])
def test_unet_engine_host_logic_vs_reference_golden(name):
    """Weight repacking (conv taps, fused QKV, hoisted K|V, GEGLU interleave, stacked time-embedding projections,
    LayerNorm folded into the consumer GEMM with row statistics from the producer, head-dim padding for tiny_15h) and the
    launch order of the whole UNet forward."""
    from b200forge.unet_engine import UNetEngine
    g = _gold(f"unet_{name}.pt")
    cfg = CF.CONFIGS[name]
    eng = UNetEngine(cfg, OU.random_state_dict(cfg, seed=g["weight_seed"]), dtype=F32, device="cpu")
    out = eng.forward(g["x"], g["t"], g["context"], g["y"])
    assert_close(f"emulated UNetEngine {name} vs reference golden", out, g["out"], max_abs=3e-4)


@pytest.mark.parametrize("sampler,key,sig", [("euler_a", "euler_a", "sigmas_auto"), ("euler", "euler", "sigmas_auto"),
                                             ("dpmpp_2m", "dpmpp_2m", "sigmas_karras")])
def test_pipeline_host_logic_vs_reference_trajectory(sampler, key, sig):
    """Txt2ImgPipeline.sample: [uncond | cond] batching, K|V cache per job, sigma / timestep tables, plans and the fused
    step, against the reference's own k-diffusion loops (CFG 7, injected noise)."""
    from b200forge.pipeline import Txt2ImgPipeline
    g = _gold("traj_tiny_xl.pt")
    cfg = CF.CONFIGS[g["config"]]
    pipe = Txt2ImgPipeline(cfg, OU.random_state_dict(cfg, seed=g["weight_seed"]), dtype=F32, device="cpu", use_graph=False)
    x = pipe.sample(g["cond"], g["uncond"], g["noise0"], sampler=sampler, cfg_scale=g["cfg_scale"], sigmas=g[sig],
                    step_noise=g["euler_a_step_noise"] if sampler == "euler_a" else None)
    assert_close(f"emulated pipeline {sampler} vs reference trajectory", x, g[key], rel_rms=2e-4)
    if sampler == "euler":  # Forge's "SGM noise multiplier" option: start = noise * sqrt(1 + sigma_0^2)
        xs = pipe.sample(g["cond"], g["uncond"], g["noise0"], sampler="euler", cfg_scale=g["cfg_scale"], sigmas=g[sig],
                         sgm_noise_multiplier=True)
        assert_close("emulated pipeline euler, sgm_noise_multiplier, vs reference trajectory", xs, g["euler_sgm"], rel_rms=2e-4)


def test_vae_engines_host_logic_vs_reference_golden():
    from b200forge.vae_engine import VAEDecoderEngine, VAEEncoderEngine
    g = _gold("vae_tiny.pt")
    cfg = CF.VAE_CONFIGS[g["config"]]
    dec = VAEDecoderEngine(cfg, OV.random_state_dict(cfg, seed=g["weight_seed"]), dtype=F32, device="cpu")
    img = dec.decode(g["z"])
    assert_close("emulated VAE decoder vs reference golden", img, torch.clamp((g["out"] + 1.0) / 2.0, 0.0, 1.0).movedim(1, -1), max_abs=1e-4)
    e = _gold("vae_enc_tiny.pt")
    enc = VAEEncoderEngine(cfg, OV.random_encoder_state_dict(cfg, seed=e["weight_seed"]), dtype=F32, device="cpu")
    assert_close("emulated VAE encoder sample vs reference golden", enc.encode(e["pixels"], e["noise"]), e["sample"], max_abs=1e-4)
    assert_close("emulated VAE encoder latent vs reference golden", enc.encode(e["pixels"], e["noise"], process_in=True), e["latent"], max_abs=1e-4)


@pytest.mark.parametrize("fname", ["flux_tiny.pt", "flux_tiny_seg.pt", "flux_tiny_odd.pt"])
def test_flux_engine_host_logic_vs_reference_golden(fname):
    """Stacked modulation GEMM and its offsets, joint [txt | img] activation, two-segment GEMMs vs per-stream launches,
    QK-norm / RoPE tables, gated in-place residuals, [qkv | mlp] split of the single-stream blocks, final layer."""
    from b200forge.flux_engine import FluxEngine
    g = _gold(fname)
    cfg = OF.CONFIGS[g["config"]]
    eng = FluxEngine(cfg, OF.random_state_dict(cfg, seed=g["weight_seed"]), dtype=F32, device="cpu")
    out = eng.forward(g["x"], g["t"], g["context"], g["y"], g["guidance"])
    assert_close(f"emulated FluxEngine {fname} vs reference golden", out, g["out"], max_abs=3e-4)


def test_flux_pipeline_host_logic_vs_oracle_loop():
    from b200forge.pipeline import FluxTxt2ImgPipeline
    cfg = OF.TINY_FLUX
    sd = OF.random_state_dict(cfg, seed=31)
    pipe = FluxTxt2ImgPipeline(cfg, sd, dtype=F32, device="cpu", use_graph=False)
    g = torch.Generator().manual_seed(32)
    B, hw, Lt, steps = 2, 16, 64, 3
    noise = torch.randn(B, 16, hw, hw, generator=g)
    cond = dict(crossattn=torch.randn(B, Lt, cfg["context_in_dim"], generator=g), vector=torch.randn(B, cfg["vec_in_dim"], generator=g))
    x = pipe.sample(cond, noise, steps=steps, guidance=4.0)
    sig = S.simple_scheduler(steps, S.flux_sigma_table(seq_len=(hw // 2) ** 2))
    gd = torch.full((B,), 4.0)

    def model(xx, sigma):
        with torch.no_grad():
            v = OF.flux_forward(sd, cfg, xx, sigma, cond["crossattn"], cond["vector"], gd)
        return S.const_denoised(xx, v, sigma.view(-1, 1, 1, 1))

    ref = S.sample_euler(model, S.const_noise_scaling(float(sig[0]), noise, torch.zeros_like(noise)), sig)
    assert_close("emulated Flux pipeline vs oracle Euler loop", x, ref, rel_rms=2e-4)


def test_v_prediction_pipeline_host_logic_vs_reference_trajectory():
    """SD2.x-style model through the public pipeline: 4-level linear-transformer UNet without label embedding,
    prediction_type="v_prediction" (the fused step's prediction switch), Euler, CFG 6 — against the reference's own run."""
    from b200forge.pipeline import Txt2ImgPipeline
    g = _gold("traj_tiny_21_v.pt")
    cfg = CF.CONFIGS[g["config"]]
    pipe = Txt2ImgPipeline(cfg, OU.random_state_dict(cfg, seed=g["weight_seed"]), dtype=F32, device="cpu", use_graph=False,
                           prediction_type="v_prediction")
    dens = []
    x = pipe.sample(g["cond"], g["uncond"], g["noise0"], sampler="euler", cfg_scale=g["cfg_scale"], sigmas=g["sigmas"],
                    callback=lambda i, xb, d: dens.append(d.clone()))
    assert_close("emulated v-pred first denoised vs reference", dens[0], g["denoised0"], rel_rms=2e-5)
    assert_close("emulated v-pred pipeline vs reference trajectory", x, g["euler"], rel_rms=2e-4)


# --------------------------------------------------------------------------------------------------------------------
# Plug points against what the UNMODIFIED reference hands them (tests/golden/plugin_calls.pt, module_calls.pt, recorded by
# oracle/gen_golden.py): P3 gets the exact argument dict backend.sampling.sampling_function.sampling_function_inner passes to
# model_options['model_function_wrapper'] (sampling_function.py:270-273) and must return what the reference's own
# apply_model returned for it; P1 / P2 get the reference models' attention calls and operator modules.  (CPU: the engines
# and operators run on the emulated ops.)
class _RecordedPredictor:
    """The reference predictor of a recorded P3 call: its prediction type, and timestep() as it evaluated for that call."""

    def __init__(self, rec):
        self.prediction_type, self._sigma, self._t = rec["prediction_type"], rec["args"]["timestep"], rec["timestep_from_sigma"]

    def timestep(self, sigma):
        assert torch.equal(sigma, self._sigma)
        return self._t


def _reference_apply_model(*a, **kw):
    raise AssertionError("the wrapper handed the call back to the reference's apply_model")


def test_p3_unet_wrapper_inside_the_reference_sampling_function(monkeypatch):
    from b200forge import plugin
    from b200forge.unet_engine import UNetEngine
    monkeypatch.setattr(plugin, "_on_device", lambda t: True)
    rec = _gold("plugin_calls.pt")["p3_unet"]
    cfg = CF.CONFIGS[rec["config"]]
    w = plugin.UNetWrapper(UNetEngine(cfg, OU.random_state_dict(cfg, seed=rec["weight_seed"]), dtype=F32, device="cpu"),
                           _RecordedPredictor(rec))
    with torch.no_grad():
        out = w(_reference_apply_model, rec["args"])
    assert w.calls_fast == 1 and w.calls_reference == 0
    assert_close("fused UNet wrapper vs the reference's apply_model for the same call", out, rec["out"], rel_rms=1e-5)


def test_p3_flux_wrapper_inside_the_reference_sampling_function(monkeypatch):
    from b200forge import plugin
    from b200forge.flux_engine import FluxEngine
    monkeypatch.setattr(plugin, "_on_device", lambda t: True)
    rec = _gold("plugin_calls.pt")["p3_flux"]
    cfg = OF.CONFIGS[rec["config"]]
    w = plugin.FluxWrapper(FluxEngine(cfg, OF.random_state_dict(cfg, seed=rec["weight_seed"]), dtype=F32, device="cpu"),
                           _RecordedPredictor(rec))
    with torch.no_grad():
        out = w(_reference_apply_model, rec["args"])
    assert w.calls_fast == 1 and w.calls_reference == 0
    assert_close("fused Flux wrapper vs the reference's apply_model for the same call", out, rec["out"], rel_rms=1e-5)


def test_p1_attention_operator_inside_the_reference_models(monkeypatch):
    """plugin.install_attention() rebinds the by-value imports of attention_function in the reference's model files
    (backend/nn/unet.py:5, flux.py:11); every distinct attention call the reference UNet (Dh = 64, [b, L, H*Dh] layout) and
    Flux transformer (Dh = 128, skip_reshape layout) make, replayed through the rebound names on seeded inputs of the same
    shapes, must run the B200 operator and reproduce the reference's result.  (CPU: the operator's kernels are the emulated
    ops; the device / dtype gate is opened for the test.)"""
    from b200forge import attention as A
    from b200forge import ops, plugin
    rec = _gold("plugin_calls.pt")
    calls = {"n": 0}
    real_attn, real_single = A.attention_function, A.attention_function_single_head_spatial

    def supports(q, k, v, heads, mask, skip_reshape):
        return mask is None and (q.shape[-1] if skip_reshape else q.shape[-1] // heads) in A.SUPPORTED_HEAD_DIMS

    monkeypatch.setattr(A, "supports", supports)
    orig_attention = ops_emulator.attention

    def counting_attention(*a, **kw):
        calls["n"] += 1
        return orig_attention(*a, **kw)

    monkeypatch.setattr(ops, "attention", counting_attention)

    def attention_pytorch(*a, **kw):
        raise AssertionError("deferred to the reference attention")

    for name in ["backend.attention"] + rec["attention_importers"]:
        monkeypatch.setitem(sys.modules, name, types.ModuleType(name))
        sys.modules[name].attention_function = attention_pytorch
    sys.modules["backend.attention"].attention_function_single_head_spatial = attention_pytorch
    plugin.install_attention()
    try:
        for key, module in (("unet_attention_calls", "backend.nn.unet"), ("flux_attention_calls", "backend.nn.flux")):
            fn = sys.modules[module].attention_function
            assert fn is A.attention_function and rec[key]
            for c in rec[key]:
                q, k, v = seeded_inputs(c["shapes"], c["seed"])
                n0 = calls["n"]
                with torch.no_grad():
                    out = fn(q, k, v, c["heads"], *c["args"], **c["kwargs"])
                assert calls["n"] == n0 + 1 and tuple(out.shape) == c["out_shape"]
                assert_close(f"reference {module} attention call {c['shapes']} through the B200 operator",
                             out.reshape(-1)[sample_index(out.numel(), c["seed"])], c["out_sample"], max_abs=5e-5)
    finally:
        plugin.uninstall_attention()
    assert A.attention_function is real_attn and A.attention_function_single_head_spatial is real_single


def _replay_module_calls(model, state_dict):
    """Build each distinct operator module the reference model runs from B200Operations with the reference's constructor
    arguments and weights, and run it on a seeded input of the recorded shape: it must reproduce the reference module's
    output.  Returns the module kinds seen in the whole recorded forward."""
    from b200forge import operations as P2
    rec = _gold("module_calls.pt")[model]
    kinds = set()
    for c in rec["calls"]:
        kinds.add(c["kind"])
        mod = getattr(P2.B200Operations, c["kind"])(**c["kwargs"])
        own = {k[len(c["name"]) + 1:]: v for k, v in state_dict.items() if k.startswith(c["name"] + ".")}
        mod.load_state_dict(own, strict=True)  # the oracle state dict names every parameter of every recorded module
        if "seed" not in c:
            continue
        x, = seeded_inputs((c["x_shape"],), c["seed"])
        with torch.no_grad():
            out = mod(x)
        assert tuple(out.shape) == c["out_shape"]
        assert_close(f"{model} {c['name']} ({c['kind']}) built from B200Operations",
                     out.reshape(-1)[sample_index(out.numel(), c["seed"])], c["out_sample"], max_abs=5e-5)
    return kinds


def _count_ops(monkeypatch, names):
    from b200forge import ops
    counted = dict.fromkeys(names, 0)
    for name in names:
        fn = getattr(ops, name)

        def wrap(*a, _fn=fn, _k=name, **kw):
            counted[_k] += 1
            return _fn(*a, **kw)
        monkeypatch.setattr(ops, name, wrap)
    return counted


def test_p2_operator_classes_inside_the_reference_unet(monkeypatch):
    """backend.operations.using_forge_operations(operations=B200Operations) (backend/operations.py:441-467): the
    reference constructs its UNet from our Linear / Conv2d / GroupNorm / LayerNorm modules.  Their NCHW / [.., C] boundary
    conversions and routing (3x3 stride 1 -> implicit GEMM, stride 2 -> im2col + GEMM, 1x1 -> GEMM) must reproduce the
    reference's modules, each built with the reference's constructor arguments.  (CPU: emulated kernels, device / dtype
    gate opened for the test.)"""
    from b200forge import operations as P2
    monkeypatch.setattr(P2, "_fast", lambda x, w: w.dtype == x.dtype)
    monkeypatch.setattr(P2, "DEFERRED", 0)
    counted = _count_ops(monkeypatch, ["gemm", "conv3x3_any", "im2col3x3", "groupnorm"])
    rec = _gold("module_calls.pt")["unet"]
    cfg = CF.CONFIGS[rec["config"]]
    kinds = _replay_module_calls("unet", OU.random_state_dict(cfg, seed=rec["weight_seed"]))
    assert kinds == {"Linear", "Conv2d", "GroupNorm", "LayerNorm"}
    assert all(counted.values()), counted


def test_hires_fix_host_logic_vs_oracle_composition():
    """Latent hires fix = first pass, torch interpolate (as the reference, modules/processing.py:1458), img2img second pass
    over the sliced schedule (sd_samplers_kdiffusion.py:136-194) — against the same composition of oracle loops."""
    from b200forge.pipeline import Txt2ImgPipeline
    cfg = CF.CONFIGS["tiny_xl"]
    sd = OU.random_state_dict(cfg, seed=1)
    pipe = Txt2ImgPipeline(cfg, sd, dtype=F32, device="cpu", use_graph=False)
    g = torch.Generator().manual_seed(21)
    B, steps, hr_steps, strength = 1, 4, 6, 0.5
    noise, noise_hr = torch.randn(B, 4, 16, 16, generator=g), torch.randn(B, 4, 32, 32, generator=g)
    cond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g), vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    uncond = dict(crossattn=torch.randn(B, 77, cfg["context_dim"], generator=g), vector=torch.randn(B, cfg["adm_in_channels"], generator=g))
    out = pipe.hires_fix(cond, uncond, noise, noise_hr, steps=steps, hr_steps=hr_steps, denoising_strength=strength,
                         sampler="euler", cfg_scale=5.0)
    pred = S.EpsPrediction()
    den = S.Denoiser(lambda xc, t, c, y: OU.unet_forward(sd, cfg, xc, t, c, y), pred, cond, uncond, 5.0)
    with torch.no_grad():
        s1 = S.get_sigmas_uniform(pred, steps)
        first = S.sample_euler(den, noise * s1[0], s1)  # txt2img start, sgm_noise_multiplier off (Forge default)
        up = torch.nn.functional.interpolate(first, size=(32, 32), mode="bilinear", antialias=False)
        s2 = S.get_sigmas_uniform(pred, hr_steps)
        sched = s2[hr_steps - int(min(strength, 0.999) * hr_steps) - 1:]
        ref = S.sample_euler(den, noise_hr * sched[0] + up, sched)
    assert out.shape == (B, 4, 32, 32)
    assert_close("emulated hires fix vs oracle composition", out, ref, rel_rms=2e-4)


def test_img2img_accepts_the_buffer_returned_by_sample():
    """sample() returns its graph's static latent buffer; feeding it straight back as img2img's init latent at the same
    size must not read the buffer after it was overwritten with the new noise."""
    from b200forge.pipeline import Txt2ImgPipeline
    cfg = CF.CONFIGS["tiny_xl"]
    pipe = Txt2ImgPipeline(cfg, OU.random_state_dict(cfg, seed=1), dtype=F32, device="cpu", use_graph=False)
    g = torch.Generator().manual_seed(23)
    noise, noise2 = torch.randn(1, 4, 16, 16, generator=g), torch.randn(1, 4, 16, 16, generator=g)
    cond = dict(crossattn=torch.randn(1, 77, cfg["context_dim"], generator=g), vector=torch.randn(1, cfg["adm_in_channels"], generator=g))
    lat = pipe.sample(cond, None, noise, steps=2, sampler="euler", cfg_scale=1.0)
    keep = lat.clone()
    a = pipe.img2img(cond, None, lat, noise2, steps=4, denoising_strength=0.5, sampler="euler", cfg_scale=1.0).clone()
    b = pipe.img2img(cond, None, keep, noise2, steps=4, denoising_strength=0.5, sampler="euler", cfg_scale=1.0)
    assert torch.equal(a, b)


def test_chroma_engine_host_logic_vs_reference_golden():
    """Chroma = the Flux block sequence fed by the Approximator's modulation vectors (backend/nn/chroma.py): the vector
    order of distribute_modulations, the [timestep | zero guidance | index] input, the residual RMSNorm-MLP stack."""
    from b200forge.flux_engine import ChromaEngine
    from oracle import chroma as OC
    g = _gold("chroma_tiny.pt")
    cfg = OC.CONFIGS[g["config"]]
    eng = ChromaEngine(cfg, OC.random_state_dict(cfg, seed=g["weight_seed"]), dtype=F32, device="cpu")
    out = eng.forward(g["x"], g["t"], g["context"])
    assert_close("emulated ChromaEngine vs reference golden", out, g["out"], max_abs=3e-4)


def test_unet_engine_control_residuals_vs_reference_golden(monkeypatch):
    """ControlNet / T2I-Adapter residuals added inside the fused forward (apply_control, backend/nn/unet.py:44-52): order
    of consumption, a None entry, NCHW residuals onto channels-last activations, skips carrying the input residuals — and
    the P3 wrapper passing `c["control"]` through (B200_CONTROL=0: it defers)."""
    from b200forge import plugin
    from b200forge.unet_engine import UNetEngine
    g = _gold("unet_tiny_xl_control.pt")
    cfg = CF.CONFIGS[g["config"]]
    sd = OU.random_state_dict(cfg, seed=g["weight_seed"])
    eng = UNetEngine(cfg, sd, dtype=F32, device="cpu")
    out = eng.forward(g["x"], g["t"], g["context"], g["y"], control=g["control"])
    assert_close("emulated UNetEngine + control vs reference golden", out, g["out"], max_abs=3e-4)
    assert len(g["control"]["input"]) == 9
    # plug point: with the switch off the call goes to Forge's own forward, with it on the fused path takes the residuals
    monkeypatch.setattr(plugin, "_on_device", lambda t: True)
    pred = S.EpsPrediction()

    class P:
        prediction_type = "epsilon"
        timestep = staticmethod(lambda s: pred.timestep(s))

    w = plugin.UNetWrapper(eng, P())
    x = torch.randn(2, 4, 16, 16, generator=torch.Generator().manual_seed(3)) * 3
    sigma = torch.tensor([4.0, 0.5])
    c = {"c_crossattn": g["context"], "y": g["y"], "control": g["control"], "transformer_options": {}}
    sentinel = torch.zeros(1)
    monkeypatch.setenv("B200_CONTROL", "0")
    assert w(lambda xx, ss, **kw: sentinel, {"input": x, "timestep": sigma, "c": c, "cond_or_uncond": [0]}) is sentinel
    monkeypatch.delenv("B200_CONTROL", raising=False)
    den = w(lambda xx, ss, **kw: sentinel, {"input": x, "timestep": sigma, "c": c, "cond_or_uncond": [0]})
    assert den is not sentinel and w.calls_fast == 1
    xc = pred.calculate_input(sigma, x)
    with torch.no_grad():
        eps = OU.unet_forward(sd, cfg, xc, pred.timestep(sigma).float(), g["context"], g["y"], control=g["control"])
    assert_close("P3 wrapper with control vs oracle", den, pred.calculate_denoised(sigma, eps, x), rel_rms=1e-5)


def test_p2_operator_classes_inside_the_reference_vae_and_flux(monkeypatch):
    """Same as above for the reference VAE decoder (Conv2d / GroupNorm at 3 and 4-channel edges, 1x1 attention convs) and
    the Flux transformer (Linear everywhere, LayerNorm without affine) built from B200Operations."""
    from b200forge import operations as P2
    monkeypatch.setattr(P2, "_fast", lambda x, w: w.dtype == x.dtype)
    monkeypatch.setattr(P2, "_FAST_DTYPES", (torch.float16, torch.bfloat16, torch.float32))
    rv, rf = _gold("module_calls.pt")["vae"], _gold("module_calls.pt")["flux"]
    vcfg, fcfg = CF.VAE_CONFIGS[rv["config"]], OF.CONFIGS[rf["config"]]
    assert _replay_module_calls("vae", OV.random_state_dict(vcfg, seed=rv["weight_seed"])) == {"Conv2d", "GroupNorm"}
    assert "Linear" in _replay_module_calls("flux", OF.random_state_dict(fcfg, seed=rf["weight_seed"]))


def test_flux_img2img_host_logic_vs_oracle_loop():
    from b200forge.pipeline import FluxTxt2ImgPipeline
    cfg = OF.TINY_FLUX
    sd = OF.random_state_dict(cfg, seed=31)
    pipe = FluxTxt2ImgPipeline(cfg, sd, dtype=F32, device="cpu", use_graph=False)
    g = torch.Generator().manual_seed(33)
    B, hw, Lt, steps, strength = 1, 16, 64, 6, 0.5
    noise, latent = torch.randn(B, 16, hw, hw, generator=g), torch.randn(B, 16, hw, hw, generator=g) * 0.7
    cond = dict(crossattn=torch.randn(B, Lt, cfg["context_in_dim"], generator=g), vector=torch.randn(B, cfg["vec_in_dim"], generator=g))
    x = pipe.img2img(cond, latent, noise, steps=steps, denoising_strength=strength, guidance=4.0)
    full = S.simple_scheduler(steps, S.flux_sigma_table(seq_len=(hw // 2) ** 2))
    sched = full[steps - int(min(strength, 0.999) * steps) - 1:]
    gd = torch.full((B,), 4.0)

    def model(xx, sigma):
        with torch.no_grad():
            v = OF.flux_forward(sd, cfg, xx, sigma, cond["crossattn"], cond["vector"], gd)
        return S.const_denoised(xx, v, sigma.view(-1, 1, 1, 1))

    ref = S.sample_euler(model, S.const_noise_scaling(float(sched[0]), noise, latent), sched)
    assert_close("emulated Flux img2img vs oracle loop", x, ref, rel_rms=2e-4)


def test_any_size_route_host_logic(monkeypatch):
    """B200_CONV_ROUTE=im2col: latent sizes the TMA convolution cannot tile (SDXL's non-square buckets, e.g. 152x104 and its /2, /4
    levels) run their 3x3 convolutions as im2col + GEMM with the same epilogue (bias, time-embedding row, residual).  Here
    a 12x20 latent (levels 12x20, 6x10, 3x5 — none of which tiles) through the UNet and VAE engines against the oracle."""
    from b200forge import ops
    from b200forge.unet_engine import UNetEngine
    from b200forge.vae_engine import VAEDecoderEngine
    cfg = CF.CONFIGS["tiny_xl"]
    sd = OU.random_state_dict(cfg, seed=1)
    eng = UNetEngine(cfg, sd, dtype=F32, device="cpu")
    assert not ops.conv3x3_supported(12, 20) and not ops.conv3x3_supported(6, 10) and not ops.conv3x3_supported(3, 5)
    monkeypatch.setenv("B200_CONV_ROUTE", "exact")
    assert not eng.supports_latent(12, 20) and eng.supports_latent(16, 16)
    monkeypatch.delenv("B200_CONV_ROUTE", raising=False)
    assert eng.supports_latent(12, 20)  # default route: generic tiling inside the implicit-GEMM kernel
    monkeypatch.setenv("B200_CONV_ROUTE", "im2col")
    assert eng.supports_latent(12, 20) and not eng.supports_latent(13, 20)  # odd sizes still need the reference's resize path
    calls = {"im2col": 0, "tma": 0}
    real_im2col, real_conv = ops.im2col3x3, ops.conv3x3

    def im2col(*a, **kw):
        calls["im2col"] += 1
        return real_im2col(*a, **kw)

    def conv(*a, **kw):
        calls["tma"] += 1
        return real_conv(*a, **kw)

    monkeypatch.setattr(ops, "im2col3x3", im2col)
    monkeypatch.setattr(ops, "conv3x3", conv)
    g = torch.Generator().manual_seed(41)
    x = torch.randn(2, 4, 12, 20, generator=g)
    ctx = torch.randn(2, 77, cfg["context_dim"], generator=g)
    y = torch.randn(2, cfg["adm_in_channels"], generator=g)
    t = torch.tensor([700.0, 40.0])
    out = eng.forward(x, t, ctx, y)
    with torch.no_grad():
        ref = OU.unet_forward(sd, cfg, x, t, ctx, y)
    assert calls["tma"] == 0 and calls["im2col"] > 20, calls
    assert_close("emulated UNetEngine at a non-tiling size vs oracle", out, ref, max_abs=3e-4)
    vcfg = CF.VAE_CONFIGS["tiny"]
    vsd = OV.random_state_dict(vcfg, seed=3)
    dec = VAEDecoderEngine(vcfg, vsd, dtype=F32, device="cpu")
    z = torch.randn(1, 4, 12, 20, generator=g) * vcfg["scaling_factor"]
    with torch.no_grad():
        vref = OV.decode_first_stage(vsd, vcfg, z)
    assert_close("emulated VAE decoder at a non-tiling size vs oracle", dec.decode(z), vref, max_abs=1e-4)


def test_p3_wrapper_follows_lora_refresh(monkeypatch):
    """Forge merges LoRA deltas into the torch module AFTER the engine was packed (backend/patcher/lora.py:352-446, hash in
    `loaded_hash`): the wrapper must re-pack (in place) when the hash changes, and hand calls back to the reference while an
    on-the-fly LoRA (`forge_online_loras`) is attached."""
    from b200forge import plugin
    from b200forge.unet_engine import UNetEngine
    monkeypatch.setattr(plugin, "_on_device", lambda t: True)
    cfg = CF.CONFIGS["tiny_xl"]
    sd = OU.random_state_dict(cfg, seed=1)

    class Layer:
        pass

    class Module:  # stands for IntegratedUNet2DConditionModel: live parameters + sub-modules
        def __init__(self):
            self.sd = {k: v.clone() for k, v in sd.items()}
            self.layers = [Layer(), Layer()]

        def state_dict(self):
            return self.sd

        def modules(self):
            return self.layers

    class Loader:
        loaded_hash = str([])

    class KModel:
        def __init__(self):
            self.diffusion_model = Module()
            self.lora_loader = Loader()

    pred = S.EpsPrediction()

    class P:
        prediction_type = "epsilon"
        timestep = staticmethod(lambda s: pred.timestep(s))

    km = KModel()
    eng = UNetEngine(cfg, km.diffusion_model.state_dict(), dtype=F32, device="cpu")
    w = plugin.UNetWrapper(eng, P(), km)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 4, 16, 16, generator=g) * 3
    sigma = torch.tensor([4.0, 0.5])
    c = {"c_crossattn": torch.randn(2, 77, cfg["context_dim"], generator=g), "y": torch.randn(2, cfg["adm_in_channels"], generator=g),
         "transformer_options": {}}
    sentinel = torch.zeros(1)
    call = lambda: w(lambda xx, ss, **kw: sentinel, {"input": x, "timestep": sigma, "c": c, "cond_or_uncond": [0]})  # noqa: E731
    base = call()
    ptr = eng.w["input_blocks.1.0.conv1.w"].data_ptr()
    # "merge a LoRA": new parameter values + a new hash, exactly what LoraLoader.refresh leaves behind
    key = "input_blocks.1.0.in_layers.2.weight"
    km.diffusion_model.sd[key] = km.diffusion_model.sd[key] + 0.05 * torch.randn(km.diffusion_model.sd[key].shape, generator=g)
    km.lora_loader.loaded_hash = str([("style.safetensors", 1.0, 1.0, False)])
    patched = call()
    assert w.weights.repacks == 1 and eng.w["input_blocks.1.0.conv1.w"].data_ptr() == ptr  # re-packed in place
    assert (patched - base).abs().max() > 1e-3, "the fused forward ignored the merged LoRA"
    xc = pred.calculate_input(sigma, x)
    with torch.no_grad():
        eps = OU.unet_forward(km.diffusion_model.sd, cfg, xc, pred.timestep(sigma).float(), c["c_crossattn"], c["y"])
    assert_close("P3 wrapper after a LoRA merge vs oracle on the patched weights", patched, pred.calculate_denoised(sigma, eps, x), rel_rms=1e-5)
    assert call() is not sentinel and w.weights.repacks == 1   # same hash: no second re-pack
    # on-the-fly LoRA: weights untouched, low-rank terms inside the layers -> reference path
    km.diffusion_model.layers[0].forge_online_loras = {"weight": []}
    km.lora_loader.loaded_hash = str([("style.safetensors", 1.0, 1.0, True)])
    assert call() is sentinel and w.calls_reference == 1
    del km.diffusion_model.layers[0].forge_online_loras
    km.lora_loader.loaded_hash = str([])
    km.diffusion_model.sd[key] = sd[key].clone()
    assert_close("P3 wrapper after the LoRA was removed", call(), base, rel_rms=1e-6)


def _forge_operations_module():
    """A stand-in for backend.operations with the behaviour of Forge's operator set that the B200 classes must keep when
    they subclass it (backend/operations.py:119-167, 442-467): Linear creates no weight until its state dict is loaded (a
    `dummy` parameter carries the storage device / dtype); every class records `parameters_manual_cast` at construction and
    then computes in the input's dtype from weights stored in another one; using_forge_operations() swaps the torch.nn
    classes for the operator set's, which is looked up as `ForgeOperations` at call time.  Each forward of the stand-in
    counts itself, so a call that reached the parent can be told apart from one the B200 class served."""
    import contextlib

    F = torch.nn.functional
    bo = types.ModuleType("backend.operations")
    bo.current_device = bo.current_dtype = None
    bo.current_manual_cast_enabled = False
    bo.parent_forwards = 0

    def cast(mod, x):
        bo.parent_forwards += 1
        if not mod.parameters_manual_cast:
            return mod.weight, mod.bias
        return mod.weight.to(x.dtype), None if mod.bias is None else mod.bias.to(x.dtype)

    class Linear(torch.nn.Module):
        def __init__(self, in_features, out_features, *args, **kwargs):
            super().__init__()
            self.in_features, self.out_features = in_features, out_features
            self.dummy = torch.nn.Parameter(torch.empty(1, device=bo.current_device, dtype=bo.current_dtype))
            self.weight = self.bias = None
            self.parameters_manual_cast = bo.current_manual_cast_enabled

        def _load_from_state_dict(self, state_dict, prefix, *args):
            if not hasattr(self, "dummy"):
                return super()._load_from_state_dict(state_dict, prefix, *args)
            for name in ("weight", "bias"):
                if prefix + name in state_dict:
                    setattr(self, name, torch.nn.Parameter(state_dict[prefix + name].to(self.dummy)))
            del self.dummy

        def forward(self, x):
            return F.linear(x, *cast(self, x))

    def storage_kwargs(kwargs):
        return dict(kwargs, device=bo.current_device, dtype=bo.current_dtype)

    class Conv2d(torch.nn.Conv2d):
        def __init__(self, *args, **kwargs):
            super().__init__(*args, **storage_kwargs(kwargs))
            self.parameters_manual_cast = bo.current_manual_cast_enabled

        def reset_parameters(self):
            return None

        def forward(self, x):
            return self._conv_forward(x, *cast(self, x))

    class GroupNorm(torch.nn.GroupNorm):
        def __init__(self, *args, **kwargs):
            super().__init__(*args, **storage_kwargs(kwargs))
            self.parameters_manual_cast = bo.current_manual_cast_enabled

        def forward(self, x):
            return F.group_norm(x, self.num_groups, *cast(self, x), self.eps)

    class LayerNorm(torch.nn.LayerNorm):
        def __init__(self, *args, **kwargs):
            super().__init__(*args, **storage_kwargs(kwargs))
            self.parameters_manual_cast = bo.current_manual_cast_enabled

        def forward(self, x):
            return F.layer_norm(x, self.normalized_shape, *cast(self, x), self.eps)

    class Embedding(torch.nn.Embedding):
        pass

    bo.ForgeOperations = type("ForgeOperations", (), dict(Linear=Linear, Conv2d=Conv2d, GroupNorm=GroupNorm, LayerNorm=LayerNorm,
                                                          Embedding=Embedding))
    names = ("Linear", "Conv2d", "GroupNorm", "LayerNorm", "Embedding")

    @contextlib.contextmanager
    def using_forge_operations(operations=None, device=None, dtype=None, manual_cast_enabled=False):
        bo.current_device, bo.current_dtype, bo.current_manual_cast_enabled = device, dtype, manual_cast_enabled
        operations = bo.ForgeOperations if operations is None else operations
        saved = {n: getattr(torch.nn, n) for n in names}
        try:
            for n in names:
                setattr(torch.nn, n, getattr(operations, n))
            yield
        finally:
            for n, cls in saved.items():
                setattr(torch.nn, n, cls)

    bo.using_forge_operations = using_forge_operations
    return bo


def test_p2_installed_operations_subclass_forges_own_classes(monkeypatch):
    """plugin.install_operations(): the hot-path classes SUBCLASS ForgeOperations' classes, so lazy weights
    (`dummy` / `_load_from_state_dict`), `parameters_manual_cast` (storage dtype != computation dtype: fp8 / bf16 storage) and
    `forge_online_loras` keep the reference's behaviour — such calls run the parent's forward (backend/operations.py:126-156).
    Forge's operator set is the stand-in above."""
    bo = _forge_operations_module()
    monkeypatch.setitem(sys.modules, "backend.operations", bo)

    from b200forge import operations as B, plugin
    forge = bo.ForgeOperations
    plugin.install_operations()
    try:
        assert issubclass(bo.ForgeOperations, forge) and issubclass(bo.ForgeOperations.Linear, forge.Linear)
        assert issubclass(bo.ForgeOperations.Conv2d, forge.Conv2d) and bo.ForgeOperations.Embedding is forge.Embedding
        with bo.using_forge_operations(device="cpu", dtype=torch.bfloat16, manual_cast_enabled=True):
            lin = torch.nn.Linear(16, 32)
            conv = torch.nn.Conv2d(8, 16, 3, padding=1)
        assert type(lin) is bo.ForgeOperations.Linear and type(conv) is bo.ForgeOperations.Conv2d
        assert isinstance(lin, forge.Linear) and lin.parameters_manual_cast and lin.weight is None  # Forge's lazy init
        g = torch.Generator().manual_seed(0)
        wl, bl = torch.randn(32, 16, generator=g).bfloat16(), torch.randn(32, generator=g).bfloat16()
        lin.load_state_dict({"weight": wl, "bias": bl})
        assert lin.weight.dtype == torch.bfloat16 and not hasattr(lin, "dummy")
        conv.load_state_dict({"weight": torch.randn(16, 8, 3, 3, generator=g).bfloat16(), "bias": torch.zeros(16).bfloat16()})
        x = torch.randn(4, 16, generator=g)  # fp32 activations on bf16 storage: manual cast in the parent's forward
        n0, p0 = B.DEFERRED, bo.parent_forwards
        y = lin(x)
        assert B.DEFERRED == n0 + 1 and bo.parent_forwards == p0 + 1 and y.dtype == torch.float32
        assert_close("manual-cast Linear through the parent's forward", y, torch.nn.functional.linear(x, wl.float(), bl.float()), max_abs=1e-5)
        assert conv(torch.randn(1, 8, 8, 8, generator=g)).dtype == torch.float32
        assert B.DEFERRED == n0 + 2 and bo.parent_forwards == p0 + 2
        lin.parameters_manual_cast = False
        assert B._plain(lin)
        lin.forge_online_loras = {}
        assert not B._plain(lin)
    finally:
        bo.ForgeOperations = plugin._installed.pop("operations")


def test_vae_tiled_decode_host_logic_vs_reference_golden():
    """VAEDecoderEngine.decode_tiled (tile walk, clamped positions, feather mask, three-pass average) and the oracle's
    restatement against the reference's own tiled_scale around its own decoder (tests/golden/vae_tiled_tiny.pt)."""
    from b200forge.vae_engine import VAEDecoderEngine
    g = _gold("vae_tiled_tiny.pt")
    cfg = CF.VAE_CONFIGS[g["config"]]
    sd = OV.random_state_dict(cfg, seed=g["weight_seed"])
    kw = dict(tile_x=g["tile_x"], tile_y=g["tile_y"], overlap=g["overlap"])
    with torch.no_grad():
        ref = OV.decode_tiled(sd, cfg, g["z"], **kw)
    assert_close("oracle tiled decode vs reference golden", ref, g["out"], max_abs=2e-5)
    dec = VAEDecoderEngine(cfg, sd, dtype=F32, device="cpu")
    img = dec.decode_tiled(g["z"], **kw)
    assert_close("emulated VAEDecoderEngine.decode_tiled vs reference golden", img, g["out"], max_abs=1e-4)
    whole = dec.decode(g["z"])
    assert (img - whole).abs().max() > 1e-3  # tiles see their own GroupNorm statistics: tiled != whole-image decode


def test_vae_decoder_16_channel_latent_with_shift_host_logic():
    """The Flux / SD3 VAE: 16 latent channels, process_out = z / scaling + shift (backend/nn/vae.py:315-316), no post-quant
    convolution — the shift is folded into the entry GEMM's bias; `processed_out=True` (the P5 contract) skips both."""
    from b200forge.vae_engine import VAEDecoderEngine
    cfg = CF.VAE_CONFIGS["tiny_flux"]
    sd = OV.random_state_dict(cfg, seed=4)
    assert "post_quant_conv.weight" not in sd
    dec = VAEDecoderEngine(cfg, sd, dtype=F32, device="cpu")
    z = torch.randn(2, 16, 12, 16, generator=torch.Generator().manual_seed(8)) * cfg["scaling_factor"]
    with torch.no_grad():
        ref = OV.decode_first_stage(sd, cfg, z)
    assert_close("emulated 16-channel VAE decoder vs oracle", dec.decode(z), ref, max_abs=1e-4)
    zz = z / cfg["scaling_factor"] + cfg["shift_factor"]
    assert_close("emulated 16-channel VAE decoder, processed-out latent", dec.decode(zz, processed_out=True), ref, max_abs=1e-4)
