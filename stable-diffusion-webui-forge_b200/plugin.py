"""Binding of the B200 backend to stable-diffusion-webui-forge's own plug points (SURVEY.md §8b, INTEGRATION.md).

    import b200forge.plugin as b200
    b200.install()                       # inside a running Forge process, after `initialize_forge()`

Nothing above `backend/` changes: `modules/processing.py` and `modules/sd_samplers_cfg_denoiser.py` keep calling
`attention_function`, `model.apply_model` (through `model_function_wrapper`), the `k_diffusion.sampling.sample_*`
names and `VAE.decode` exactly as before.

Fast-path predicate (reference hooks that the fused forward cannot honour => the call goes to the reference code):
  transformer_options has no patches / patches_replace / block_modifiers / block_inner_modifiers /
  group_norm_wrapper; control is None; no c_concat; epsilon prediction; fp16/bf16 computation dtype; CUDA sm_100.
"""
from __future__ import annotations

import sys
from typing import Any, Callable, Dict, Optional

import torch

from . import attention as b200_attention
from . import k_samplers, ops
from .unet_engine import UNetEngine

_BLOCKING_KEYS = ("patches", "patches_replace", "block_modifiers", "block_inner_modifiers", "group_norm_wrapper")
# modules that imported attention_function *by value* (backend/nn/unet.py:5, nn/flux.py:11, nn/chroma.py:10, nn/vae.py:3)
_ATTENTION_IMPORTERS = ("backend.nn.unet", "backend.nn.flux", "backend.nn.chroma", "backend.nn.mmditx")
_installed: Dict[str, Any] = {}


def _on_device(t: torch.Tensor) -> bool:
    """The fused path serves CUDA tensors only (one seam, so the CPU wiring tests can stand an emulation in)."""
    return t.is_cuda


def fast_path_ok(c: dict) -> bool:
    """True when the conditioning dict of one apply_model call can be served by the fused forward."""
    to = c.get("transformer_options") or {}
    for k in _BLOCKING_KEYS:
        v = to.get(k)
        if v:
            return False
    if c.get("c_concat") is not None:
        return False
    if c.get("control") is not None and not _control_ok(c["control"]):
        return False
    return c.get("c_crossattn") is not None


def _control_ok(control) -> bool:
    """ControlNet / T2I-Adapter residuals the fused UNet can add itself (UNetEngine.forward_cols(control=...)): a dict of
    lists of CUDA tensors / None under the reference's three names (backend/nn/unet.py:44-52); their shapes (the
    activation's, with its batch or batch 1) are checked against the latent by UNetEngine.control_fits.  B200_CONTROL=0
    sends such calls to Forge's own forward instead."""
    import os
    if os.environ.get("B200_CONTROL") == "0" or not isinstance(control, dict):
        return False
    for k, lst in control.items():
        if k not in ("input", "middle", "output") or not isinstance(lst, (list, tuple)):
            return False
        if any(t is not None and not (torch.is_tensor(t) and t.dim() == 4) for t in lst):
            return False
    return True


# ------------------------------------------------------------------------------------------------- P1 attention
def install_attention(modules: Optional[dict] = None) -> None:
    """Rebind `attention_function` (+ the single-head VAE variant) in backend.attention and in every module that
    imported it by value; the originals are kept as the fallback for masks / unsupported head dims."""
    mods = sys.modules if modules is None else modules
    ba = mods.get("backend.attention")
    if ba is None:
        raise RuntimeError("backend.attention is not imported — call install() from inside Forge")
    if "attention" not in _installed:
        _installed["attention"] = (ba.attention_function, ba.attention_function_single_head_spatial)
    b200_attention.fallback, b200_attention.fallback_single_head = _installed["attention"]
    ba.attention_function = b200_attention.attention_function
    ba.attention_function_single_head_spatial = b200_attention.attention_function_single_head_spatial
    for name in _ATTENTION_IMPORTERS:
        m = mods.get(name)
        if m is not None and hasattr(m, "attention_function"):
            m.attention_function = b200_attention.attention_function
    v = mods.get("backend.nn.vae")
    if v is not None and hasattr(v, "attention_function_single_head_spatial"):
        v.attention_function_single_head_spatial = b200_attention.attention_function_single_head_spatial


def uninstall_attention(modules: Optional[dict] = None) -> None:
    mods = sys.modules if modules is None else modules
    if "attention" not in _installed:
        return
    fn, fn1 = _installed.pop("attention")
    ba = mods.get("backend.attention")
    if ba is not None:
        ba.attention_function, ba.attention_function_single_head_spatial = fn, fn1
    for name in _ATTENTION_IMPORTERS:
        m = mods.get(name)
        if m is not None and hasattr(m, "attention_function"):
            m.attention_function = fn
    v = mods.get("backend.nn.vae")
    if v is not None and hasattr(v, "attention_function_single_head_spatial"):
        v.attention_function_single_head_spatial = fn1
    b200_attention.fallback = b200_attention.fallback_single_head = None


# ------------------------------------------------------------------------------------------------- P2 operators
def install_operations(modules: Optional[dict] = None) -> None:
    """Make `using_forge_operations(operations=None)` (backend/loader.py:159) build models from B200Operations:
    the default operator set is looked up as `backend.operations.ForgeOperations` at call time (:447-453)."""
    from .operations import make_operations
    mods = sys.modules if modules is None else modules
    bo = mods.get("backend.operations")
    if bo is None:
        raise RuntimeError("backend.operations is not imported")
    if "operations" not in _installed:
        _installed["operations"] = bo.ForgeOperations
    # the four hot-path classes subclass Forge's own (lazy weights, manual cast, online LoRA keep working: whatever the
    # fused kernels do not cover runs the parent's forward), every other attribute is inherited
    bo.ForgeOperations = make_operations(_installed["operations"])


# ------------------------------------------------------------------------------------------------- P3 whole model
class _WeightTracker:
    """Keeps an engine's packed weights in step with the torch module Forge patches.

    Forge applies LoRA per generation, after the model (and this plug-in's engine) was built: `networks.load_networks`
    clones the patcher (the clone keeps `model_options`, so the wrapper survives), `ModelPatcher.refresh_loras`
    (backend/patcher/base.py:125-126) calls `LoraLoader.refresh` (backend/patcher/lora.py:352-446), which either MERGES the
    deltas into fresh Parameters of the module or — `online_mode` — attaches `forge_online_loras` to the layers and leaves the
    weights alone; `loaded_hash` names the set that is currently applied.  So before every fused forward:
      * hash changed            -> re-pack the engine from the module's live state dict (in place: buffers keep their
                                   addresses, so captured CUDA graphs stay valid);
      * any online LoRA present -> not servable by the fused forward (low-rank terms inside every Linear): reference path.
    A module without a `lora_loader` (standalone use, tests) is treated as never patched."""

    def __init__(self, engine, owner, module):
        self.engine, self.owner, self.module = engine, owner, module
        self.packed_hash = self._hash()
        self.online = self._has_online()
        self.repacks = 0

    def _hash(self):
        loader = getattr(self.owner, "lora_loader", None)
        return getattr(loader, "loaded_hash", None)

    def _has_online(self) -> bool:
        mods = getattr(self.module, "modules", None)
        return bool(mods) and any(hasattr(m, "forge_online_loras") for m in self.module.modules())

    def servable(self) -> bool:
        h = self._hash()
        if h != self.packed_hash:
            self.online = self._has_online()          # refresh() attaches / removes them together with the hash change
            self.engine.repack(self.module.state_dict())
            self.packed_hash = h
            self.repacks += 1
        return not self.online


class _GraphedApplyModel:
    """KModel.apply_model for one (batch, latent size, context length) as ONE CUDA graph with static buffers: entry scaling +
    UNet forward + eps -> denoised (backend/modules/k_model.py:25-46).  The eager forward is ~1000 ctypes launches per call;
    replaying the captured graph is what makes the plug-in path as fast as the standalone pipeline.  The engine's packed
    weights are refreshed in place on a LoRA change (`UNetEngine.repack`), so a captured graph stays valid."""

    def __init__(self, engine: UNetEngine, n: int, hh: int, ww: int, n_ctx: int, prediction: int):
        dev, dt, cfg = engine.device, engine.dtype, engine.cfg
        self.engine, self.prediction = engine, prediction
        self.x = torch.zeros((n, cfg["in_channels"], hh, ww), dtype=torch.float32, device=dev)
        self.sigma = torch.ones((n,), dtype=torch.float32, device=dev)
        self.t = torch.zeros((n,), dtype=torch.float32, device=dev)
        self.ctx = torch.zeros((n, n_ctx, cfg["context_dim"]), dtype=dt, device=dev)
        self.y = torch.zeros((n, cfg["adm_in_channels"]), dtype=dt, device=dev) if engine.has_label else None
        self.out = torch.empty_like(self.x)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):  # warm-up: first-call attribute setup, allocator pools
                self._eager()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        n0 = ops.LAUNCHES
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._eager()
        self.launches = ops.LAUNCHES - n0

    def _eager(self):
        eps = self.engine.forward_sigma(self.x, self.sigma, self.t, self.ctx, self.y, reps=1)
        ops.eps_to_denoised(self.x, eps, self.sigma, prediction=self.prediction, out=self.out)

    def __call__(self, x, sigma, t, ctx, y):
        self.x.copy_(x)
        self.sigma.copy_(sigma)
        self.t.copy_(t)
        self.ctx.copy_(ctx)
        if self.y is not None:
            self.y.copy_(y)
        self.graph.replay()
        ops.LAUNCHES += self.launches
        return self.out.clone()  # the static output buffer is overwritten by the next call


class UNetWrapper:
    """`model_options['model_function_wrapper']` (reference backend/sampling/sampling_function.py:270-273):
    wrapper(apply_model_fn, {"input": x fp32 [N,4,h,w], "timestep": sigma [N], "c": {...}, "cond_or_uncond": [...]})
    -> denoised fp32 [N,4,h,w].  Serves the call from the fused channels-last forward when `fast_path_ok`, else
    calls `apply_model_fn(input, timestep, **c)` (the reference path) unchanged."""

    def __init__(self, engine: UNetEngine, predictor, kmodel=None):
        self.engine = engine
        self.predictor = predictor  # backend.modules.k_prediction.Prediction (for .timestep and .prediction_type)
        # kmodel: the KModel whose diffusion_model Forge patches (LoRA); None = weights never change (standalone use)
        self.weights = None if kmodel is None else _WeightTracker(engine, kmodel, kmodel.diffusion_model)
        self.calls_fast = 0
        self.calls_reference = 0
        # one CUDA graph per call shape (B200_PLUGIN_GRAPH=0: eager launches); calls with control residuals stay eager
        import os
        self.use_graph = os.environ.get("B200_PLUGIN_GRAPH", "1") != "0"
        self._graphs: Dict[tuple, _GraphedApplyModel] = {}

    def __call__(self, apply_model_fn: Callable, args: dict):
        x, sigma, c = args["input"], args["timestep"], args["c"]
        ptype = getattr(self.predictor, "prediction_type", "epsilon")
        if (not fast_path_ok(c) or not _on_device(x) or x.dtype != torch.float32 or ptype not in ("epsilon", "v_prediction")
                or (self.engine.has_label and c.get("y") is None) or x.dim() != 4
                or not self.engine.supports_latent(x.shape[2], x.shape[3])
                or (c.get("control") is not None and not self.engine.control_fits(c["control"], x.shape[0], x.shape[2], x.shape[3]))
                or (self.weights is not None and not self.weights.servable())):
            self.calls_reference += 1
            return apply_model_fn(x, sigma, **c)
        self.calls_fast += 1
        eng = self.engine
        x = x.contiguous()
        sigma = sigma.float().contiguous()
        t = self.predictor.timestep(sigma).float().contiguous()           # k_model.py:35
        ctx = c["c_crossattn"].to(eng.dtype).contiguous()                  # k_model.py:36
        y = c.get("y")
        y = None if y is None else y.to(eng.dtype).contiguous()
        pred = 1 if ptype == "v_prediction" else 0
        if self.use_graph and x.is_cuda and c.get("control") is None and not torch.cuda.is_current_stream_capturing():
            key = (tuple(x.shape), ctx.shape[1], pred)
            g = self._graphs.get(key)
            if g is None:
                if len(self._graphs) >= 4:  # a handful of shapes per job (cond/uncond batched or not, hires pass)
                    self._graphs.pop(next(iter(self._graphs)))
                g = self._graphs[key] = _GraphedApplyModel(eng, x.shape[0], x.shape[2], x.shape[3], ctx.shape[1], pred)
            return g(x, sigma, t, ctx, y)
        eps = eng.forward_sigma(x, sigma, t, ctx, y, reps=1, control=c.get("control"))  # k_model.py:27,34 fused into the entry
        return ops.eps_to_denoised(x, eps, sigma, prediction=pred)  # k_model.py:45-46


def install_unet_wrapper(unet_patcher, engine: Optional[UNetEngine] = None) -> UNetWrapper:
    """Attach the fused forward to a Forge `UnetPatcher` (backend/patcher/unet.py) through its own setter
    `set_model_unet_function_wrapper` (backend/patcher/base.py:146-147)."""
    kmodel = unet_patcher.model
    dm = kmodel.diffusion_model
    if engine is None:
        cfg = dict(dm.config) if hasattr(dm, "config") else None
        if cfg is None:
            raise ValueError("pass engine=UNetEngine(cfg, state_dict) — the module carries no config")
        engine = UNetEngine(cfg, dm.state_dict(), dtype=kmodel.computation_dtype, device=unet_patcher.load_device)
    w = UNetWrapper(engine, kmodel.predictor, kmodel)
    unet_patcher.set_model_unet_function_wrapper(w)
    return w


class FluxWrapper:
    """The same plug point (P3) for Flux: KModel.apply_model with PredictionFlux ('const': model input = x, timestep =
    sigma, denoised = x - sigma * output; backend/modules/k_model.py:25-46, k_prediction.py:74-92,285-322) served by
    the fused DiT forward.  `c` carries c_crossattn (T5 states), y (pooled CLIP) and guidance
    (backend/diffusion_engine/flux.py:92)."""

    def __init__(self, engine, predictor, kmodel=None):
        self.engine = engine
        self.predictor = predictor
        self.weights = None if kmodel is None else _WeightTracker(engine, kmodel, kmodel.diffusion_model)
        self.calls_fast = 0
        self.calls_reference = 0

    def __call__(self, apply_model_fn: Callable, args: dict):
        x, sigma, c = args["input"], args["timestep"], args["c"]
        eng = self.engine
        ok = (fast_path_ok(c) and c.get("control") is None and _on_device(x) and x.dtype == torch.float32 and x.dim() == 4
              and getattr(self.predictor, "prediction_type", None) == "const" and c.get("c_concat") is None
              and c.get("y") is not None
              and (c.get("guidance") is not None or not eng.guidance_embed)
              and (self.weights is None or self.weights.servable()))
        if not ok:
            self.calls_reference += 1
            return apply_model_fn(x, sigma, **c)
        self.calls_fast += 1
        x = x.contiguous()
        sigma = sigma.float().contiguous()
        t = self.predictor.timestep(sigma).float().contiguous()
        g = c.get("guidance")
        g = None if g is None else g.to(x.device).float().contiguous()
        ctx, y = c["c_crossattn"].to(eng.dtype).contiguous(), c["y"].to(eng.dtype).contiguous()
        if (x.shape[2] | x.shape[3]) & 1:  # odd latent: the engine pads circularly and crops (flux.py:394-397, 412)
            out = ops.nchw_to_nhwc(eng.forward(x, t, ctx, y, g), eng.dtype)
        else:
            out = eng.forward_nhwc(x, t, ctx, y, g)
        return ops.eps_to_denoised(x, out, sigma, prediction=0)  # x - sigma * v


def install_flux_wrapper(unet_patcher, engine=None) -> FluxWrapper:
    """Attach the fused Flux forward to a Forge `UnetPatcher` whose model is a KModel around
    IntegratedFluxTransformer2DModel (backend/diffusion_engine/flux.py)."""
    from .flux_engine import FluxEngine
    kmodel = unet_patcher.model
    dm = kmodel.diffusion_model
    if engine is None:
        cfg = dict(dm.config) if hasattr(dm, "config") else None
        if cfg is None:
            raise ValueError("pass engine=FluxEngine(cfg, state_dict) — the module carries no config")
        keys = ("in_channels", "vec_in_dim", "context_in_dim", "hidden_size", "mlp_ratio", "num_heads", "depth",
                "depth_single_blocks", "axes_dim", "theta", "qkv_bias", "guidance_embed")
        engine = FluxEngine({k: cfg[k] for k in keys}, dm.state_dict(), dtype=kmodel.computation_dtype,
                            device=unet_patcher.load_device)
    w = FluxWrapper(engine, kmodel.predictor, kmodel)
    unet_patcher.set_model_unet_function_wrapper(w)
    return w


# ------------------------------------------------------------------------------------------------- P6 ControlNet model
class ControlNetWrapper:
    """`transformer_options['controlnet_model_function_wrapper']` (set by UnetPatcher.set_controlnet_model_function_wrapper,
    backend/patcher/unet.py:169-170; copied onto every ControlNet of the chain, sampling_function.py:261-268):
    ControlNet.get_control calls wrapper(x=, hint=, timesteps=, context=, y=, model=, inner_model=) instead of
    `control_model(...)` (backend/patcher/controlnet.py:329-339) and hands the result to control_merge, which keeps strength,
    per-block / per-sigma weighting, masks, global average pooling and the merging of several ControlNets.

    One ControlNetEngine per control model (built on its first fast call from `inner_model.state_dict()`).  A call is
    handed back exactly as get_control's own no-wrapper branch would run it when it is a T2I-Adapter call
    (`inner_t2i_model`, controlnet.py:524-531), a Control-LoRA, on a tensor that is not on CUDA, in a dtype other than
    fp16 / bf16, at a latent size the engine does not tile, with a hint that is not 8x the latent, for a model whose
    engine could not be built (B200_STRICT=1: that raises instead), or when B200_CONTROLNET=0.  What is decided per
    model (Control-LoRA or not, engine built or not) is decided once, on its first call."""

    def __init__(self):
        import weakref
        self.engines = weakref.WeakKeyDictionary()  # inner_model -> ControlNetEngine
        self.unserved = weakref.WeakKeyDictionary()  # inner_model -> why its calls go back to Forge (Control-LoRA, build error)
        self.calls_fast = 0
        self.calls_reference = 0

    @staticmethod
    def _is_control_lora(model, inner_model) -> bool:
        if type(model).__name__ == "ControlLora":
            return True
        mods = getattr(inner_model, "modules", None)
        return mods is not None and any(hasattr(m, "up") and hasattr(m, "down") for m in inner_model.modules())

    def _engine(self, model, inner_model, x):
        """The engine of `inner_model` in x's dtype on x's device, or None when its calls go back to Forge."""
        import os
        from .controlnet_engine import ControlNetEngine, controlnet_config
        if inner_model in self.unserved:
            return None
        eng = self.engines.get(inner_model)
        if eng is None or eng.dtype != x.dtype or eng.device != x.device:
            if self._is_control_lora(model, inner_model):
                self.unserved[inner_model] = "Control-LoRA"
                return None
            try:
                eng = ControlNetEngine(controlnet_config(inner_model), inner_model.state_dict(), dtype=x.dtype, device=x.device)
            except Exception as e:
                if os.environ.get("B200_STRICT") == "1":
                    raise
                self.unserved[inner_model] = f"engine not built: {type(e).__name__}: {e}"
                return None
            self.engines[inner_model] = eng
        return eng

    def __call__(self, x=None, hint=None, timesteps=None, context=None, y=None, model=None, inner_model=None, **kw):
        import os
        if "inner_t2i_model" in kw:  # T2I-Adapter: runs once per job on the hint alone (controlnet.py:531)
            self.calls_reference += 1
            dev = getattr(model, "device", None)
            return inner_model(hint if dev is None else hint.to(dev))
        tensors = [x, timesteps, context] + ([] if y is None else [y])
        eng = None
        if (os.environ.get("B200_CONTROLNET") != "0" and type(model).__name__ != "ControlLora"
                and all(torch.is_tensor(t) and _on_device(t) for t in tensors) and torch.is_tensor(hint)
                and x.dim() == 4 and x.dtype in (torch.float16, torch.bfloat16)):
            eng = self._engine(model, inner_model, x)
            if eng is not None and not (eng.supports_latent(x.shape[2], x.shape[3]) and eng.supports_hint(hint, x.shape[0], x.shape[2], x.shape[3])
                    and (y is not None or not eng.has_label)):
                eng = None
        if eng is None:
            self.calls_reference += 1
            dev = getattr(model, "device", None)
            return inner_model(x=x, hint=hint if dev is None else hint.to(dev), timesteps=timesteps, context=context, y=y)
        self.calls_fast += 1
        return eng.forward(x, hint, timesteps, context, y)


def install_controlnet_wrapper(unet_patcher) -> ControlNetWrapper:
    """Serve every ControlNet model of the jobs this UnetPatcher runs from the fused engine (P6).  The wrapper lives in
    the patcher's transformer_options, so clones made per generation (LoRA, ControlNet units) inherit it."""
    w = ControlNetWrapper()
    unet_patcher.set_controlnet_model_function_wrapper(w)
    return w


# ------------------------------------------------------------------------------------------------- P4 samplers
_SAMPLER_NAMES = ("sample_euler", "sample_euler_ancestral", "sample_dpmpp_2m", "sample_heun", "sample_dpm_2",
                  "sample_dpm_2_ancestral", "sample_dpmpp_2s_ancestral", "sample_lms", "sample_dpmpp_sde",
                  "sample_dpmpp_2m_sde", "sample_dpmpp_3m_sde", "sample_heunpp2", "sample_ipndm", "sample_ipndm_v", "sample_deis")


def install_extra_samplers(modules: Optional[dict] = None) -> None:
    """Forge's own extra samplers are plain functions referenced from sampler tables: Restart
    (modules/sd_samplers_extra.py:7, table entry modules/sd_samplers_kdiffusion.py:38) and LCM (modules/sd_samplers_lcm.py:68,
    :100).  Rebinding the module attribute before the tables are built (or patching the table entry) swaps them."""
    mods = sys.modules if modules is None else modules
    ex = mods.get("modules.sd_samplers_extra")
    if ex is not None and hasattr(ex, "restart_sampler"):
        if "restart" not in _installed:
            _installed["restart"] = ex.restart_sampler
        k_samplers.reference_restart_sampler = _installed["restart"]
        ex.restart_sampler = k_samplers.restart_sampler
    lcm = mods.get("modules.sd_samplers_lcm")
    if lcm is not None and hasattr(lcm, "sample_lcm"):
        if "lcm" not in _installed:
            _installed["lcm"] = lcm.sample_lcm
        k_samplers.reference_sample_lcm = _installed["lcm"]
        lcm.sample_lcm = k_samplers.sample_lcm


def install_samplers(modules: Optional[dict] = None) -> None:
    """Replace the k_diffusion.sampling functions that have a fused version (Euler, Euler a, DPM++ 2M, Heun, DPM2, DPM2 a,
    DPM++ 2S a): the sampler table (modules/sd_samplers_kdiffusion.py:14-41) resolves them by getattr at sampler
    construction (:76).  The originals stay reachable as `k_samplers.reference_<name>` for the cases handed back."""
    mods = sys.modules if modules is None else modules
    ks = mods.get("k_diffusion.sampling")
    if ks is None:
        raise RuntimeError("k_diffusion.sampling is not imported")
    if "samplers" not in _installed:
        _installed["samplers"] = {n: getattr(ks, n) for n in _SAMPLER_NAMES if hasattr(ks, n)}
    for n, fn in _installed["samplers"].items():
        setattr(k_samplers, "reference_" + n, fn)
        setattr(ks, n, getattr(k_samplers, n))


# ------------------------------------------------------------------------------------------------- P5 VAE
class VAEDecodeWrapper:
    """`model_options['model_vae_decode_wrapper']` (reference backend/patcher/vae.py:150-155):
    wrapper(decode_inner_fn, samples_in [B,4,h,w]) -> images [B,H,W,3] fp32 in [0,1] on the output device.
    NB: Forge hands this wrapper the *processed-out* latent (engine.decode_first_stage applies z / scaling + shift first,
    diffusion_engine/sdxl.py:134-138), so the engine is told not to apply process_out again."""

    def __init__(self, vae_engine, output_device=None, vae_module=None):
        self.engine = vae_engine
        self.output_device = output_device
        # vae_module: the torch VAE Forge may patch (it wraps it in a ModelPatcher too, backend/patcher/vae.py:60-75)
        self.weights = None if vae_module is None else _WeightTracker(vae_engine, vae_module, vae_module)

    def decode_tiled(self, samples_in: torch.Tensor, tile_x: int = 64, tile_y: int = 64, overlap: int = 16) -> torch.Tensor:
        """VAE.decode_tiled (backend/patcher/vae.py:157-160): same contract (processed-out latent in, NHWC images out)."""
        img = self.engine.decode_tiled(samples_in.to(self.engine.device).float().contiguous(), tile_x, tile_y, overlap,
                                       processed_out=True)
        return img if self.output_device is None else img.to(self.output_device)

    def __call__(self, decode_inner_fn: Callable, samples_in: torch.Tensor):
        import os
        if os.environ.get("B200_VAE_ALWAYS_TILED") == "1" and _on_device(samples_in) and samples_in.dim() == 4:
            return self.decode_tiled(samples_in)  # memory_management.VAE_ALWAYS_TILED (backend/patcher/vae.py:129-130)
        if (not _on_device(samples_in) or samples_in.dim() != 4 or not self.engine.supports_latent(samples_in.shape[2], samples_in.shape[3])
                or (self.weights is not None and not self.weights.servable())):
            return decode_inner_fn(samples_in)
        img = self.engine.decode(samples_in.float().contiguous(), processed_out=True)
        return img if self.output_device is None else img.to(self.output_device)


class VAEEncodeWrapper:
    """`model_options['model_vae_encode_wrapper']` (reference backend/patcher/vae.py:186-191):
    wrapper(encode_inner_fn, pixel_samples [B,H,W,3] in [0,1]) -> latent [B,zc,h,w] fp32 on the output device, the
    un-scaled posterior sample (the diffusion engine applies process_in afterwards, diffusion_engine/sdxl.py:128-132).
    A `model_vae_regulation` hook or a size the TMA convolution path cannot tile goes back to Forge's own encode."""

    def __init__(self, vae_engine, output_device=None, patcher=None, vae_module=None):
        self.engine = vae_engine
        self.output_device = output_device
        self.patcher = patcher
        self.weights = None if vae_module is None else _WeightTracker(vae_engine, vae_module, vae_module)

    def __call__(self, encode_inner_fn: Callable, pixel_samples: torch.Tensor):
        has_reg = self.patcher is not None and self.patcher.model_options.get("model_vae_regulation") is not None
        if (has_reg or pixel_samples.dim() != 4 or pixel_samples.shape[-1] != 3 or not torch.cuda.is_available()
                or not self.engine.supports_image(pixel_samples.shape[1], pixel_samples.shape[2])
                or (self.weights is not None and not self.weights.servable())):
            return encode_inner_fn(pixel_samples)
        z = self.engine.encode(pixel_samples.to(self.engine.device).float().contiguous())
        return z if self.output_device is None else z.to(self.output_device)


def install(modules: Optional[dict] = None, attention: bool = True, samplers: bool = True, operations: bool = False) -> None:
    """One call from inside Forge.  The per-checkpoint hooks (install_unet_wrapper, VAEDecodeWrapper) are attached when
    a model is loaded, e.g. from a `script_callbacks.on_model_loaded` callback (INTEGRATION.md)."""
    from . import lib
    lib.check(lib.load().b200_device_ok())
    if attention:
        install_attention(modules)
    if samplers:
        install_samplers(modules)
        install_extra_samplers(modules)
    if operations:
        install_operations(modules)
