"""Fused channels-last forward of the LDM ControlNet (backend/nn/cnets/cldm.py:244-270) — the model Forge's ControlNet
units run on the whole [uncond | cond] batch before every UNet call.

A ControlNet is the UNet's encoder half (input blocks + middle block, same constructor) plus a hint encoder
(`input_hint_block`: eight 3x3 convolutions from the control image down to latent resolution) and one zero-initialised
1x1 convolution per block output.  So the engine is a UNetEngine whose structure stops after the middle block: weight
packing and the ResBlock / SpatialTransformer launch sequences are the UNet's own.  On top of them:

  guided_hint    input_hint_block on the hint's own batch (usually one image), once per hint rather than once per step:
                 it reads neither the time embedding nor the context.  Each conv is im2col3x3 (stride 1 or 2) + one GEMM
                 with the SiLU in its epilogue; cached on the engine, keyed on the hint tensor's identity, version and shape.
  per step       conv_in GEMM -> += guided_hint (batch-1 broadcast, NHWC) -> encoder + middle blocks -> per block output
                 one 1x1 GEMM (zero conv, + bias) and one NHWC -> NCHW conversion into the fresh tensor Forge expects.

Cross-attention K|V is projected per call (the UNet's eager path): the ControlNet sees a new context batch every call.
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import ops
from .ops import EPI_NONE, EPI_SILU
from .unet_engine import SD, UNetEngine, encoder_structure


def hint_convs(hint_channels: int, model_channels: int):
    """(state-dict index, Cin, Cout, stride) of input_hint_block's convolutions (cldm.py:116-132); SiLU after all but the last."""
    chans = [hint_channels, 16, 16, 32, 32, 96, 96, 256, model_channels]
    strides = [1, 1, 2, 1, 2, 1, 2, 1]
    return [(2 * i, chans[i], chans[i + 1], strides[i]) for i in range(8)]


def controlnet_structure(cfg: dict) -> dict:
    inp, mid, _, ch = encoder_structure(cfg)
    return dict(input=inp, middle=mid, output=[], out_ch=ch)


def controlnet_config(module) -> dict:
    """Engine config of a live `cldm.ControlNet`.  Forge builds the module from a config it does not keep
    (modules_forge/supported_controlnet.py:111-119), so what the constructor stores as attributes is read from them
    (cldm.py:57-84) and the rest is derived from the state dict's keys and shapes.  A ControlNet without cross-attention
    (every transformer depth 0, as in some small SDXL ControlNets) has no key to read the context width or the projection
    kind from; neither is used then, and they are left None / False."""
    sd = module.state_dict()
    nrb = list(module.num_res_blocks)
    cm = list(module.channel_mult)
    mc = int(module.model_channels)
    nh, nhc = int(module.num_heads), int(module.num_head_channels)
    # transformer depth of every input block that holds a ResBlock, in constructor order (0 where it has no transformer)
    depth, i = [], 1
    for level in range(len(cm)):
        for _ in range(nrb[level]):
            depth.append(_depth(sd, f"input_blocks.{i}.1"))
            i += 1
        i += level != len(cm) - 1
    ctx_key = next((k for k in sd if k.endswith("attn2.to_k.weight")), None)
    proj = next((k for k in sd if k.endswith(".proj_in.weight")), None)
    label = "label_emb.0.0.weight" in sd
    return dict(
        in_channels=int(sd["input_blocks.0.0.weight"].shape[1]), model_channels=mc, num_res_blocks=nrb, channel_mult=cm,
        transformer_depth=depth, transformer_depth_middle=_depth(sd, "middle_block.1") if "middle_block.1.norm.weight" in sd else -1,
        num_heads=nh, num_head_channels=nhc, use_linear_in_transformer=proj is not None and sd[proj].dim() == 2,
        context_dim=None if ctx_key is None else int(sd[ctx_key].shape[1]), adm_in_channels=int(sd["label_emb.0.0.weight"].shape[1]) if label else None,
        num_classes="sequential" if label else None, hint_channels=int(sd["input_hint_block.0.weight"].shape[1]))


def _depth(sd: SD, p: str) -> int:
    d = 0
    while f"{p}.transformer_blocks.{d}.norm1.weight" in sd:
        d += 1
    return d


class ControlNetEngine(UNetEngine):
    """Packed weights + launch sequence of one ControlNet forward (`cldm.ControlNet.forward`'s contract).

    The subclass reuses UNetEngine's packing and block launch code; its structure has no decoder and no `out.*` weights,
    so the UNet-only entry points it inherits (`forward_cols`, `forward_sigma`, `cross_kv_layers` / `alloc_kv_cache` /
    `fill_kv_cache` for the per-job K|V cache) must not be called on it: `forward` is the one entry point."""

    HINT_CACHE = 4  # two ControlNet units may share one model with different hints; hires fix adds a second size

    def __init__(self, cfg: dict, state_dict: SD, dtype: torch.dtype = torch.float16, device="cuda"):
        self._hints: List[tuple] = []  # (hint tensor, (version, shape, dtype), guided_hint NHWC), most recent last
        super().__init__(cfg, state_dict, dtype, device)

    @staticmethod
    def _structure(cfg: dict) -> dict:
        return controlnet_structure(cfg)

    def repack(self, state_dict: SD) -> None:
        super().repack(state_dict)
        self._hints.clear()

    def _pack(self, sd: SD) -> None:
        w = self.w
        g = lambda k: self._t(sd[k])  # noqa: E731
        self._pack_embeddings(g)
        self._pack_blocks(g, self.st["input"] + [self.st["middle"]])
        self.hint = hint_convs(self.cfg["hint_channels"], self.mc)
        for i, cin, cout, _ in self.hint:
            wp = ops.pack_conv3x3(g(f"input_hint_block.{i}.weight"))
            kp = (wp.shape[1] + 63) // 64 * 64  # im2col columns padded to the GEMM's K granularity, as conv_in's 36 -> 64
            wk = torch.zeros((cout, kp), dtype=self.dtype, device=self.device)
            wk[:, : wp.shape[1]] = wp
            w[f"hint.{i}.w"], w[f"hint.{i}.b"] = wk, g(f"input_hint_block.{i}.bias")
        self.zero_convs = [f"zero_convs.{i}.0" for i in range(len(self.st["input"]))] + ["middle_block_out.0"]
        for p in self.zero_convs:
            wt = g(p + ".weight")
            w[p + ".w"], w[p + ".b"] = wt.reshape(wt.shape[0], wt.shape[1]).contiguous(), g(p + ".bias")

    # ------------------------------------------------------------------------------------------ hint
    def guided_hint(self, hint: torch.Tensor) -> torch.Tensor:
        """input_hint_block(hint) as NHWC [hint batch, H/8, W/8, model_channels], computed once per hint tensor: an entry
        is reused while the caller's tensor is the same object with the same version counter (an in-place edit bumps it)
        and shape."""
        key = (hint._version, tuple(hint.shape), hint.dtype)
        for i, (t, k, gh) in enumerate(self._hints):
            if t is hint and k == key:
                self._hints.append(self._hints.pop(i))
                return gh
        gh = self._hint_block(hint)
        self._hints.append((hint, key, gh))  # holding the tensor keeps its identity from being reused
        if len(self._hints) > self.HINT_CACHE:
            self._hints.pop(0)
        return gh

    def _hint_block(self, hint: torch.Tensor) -> torch.Tensor:
        w = self.w
        src = hint.to(self.device)
        if src.dtype not in (torch.float32, self.dtype):
            src = src.float()
        nh, _, H, W = src.shape
        out = torch.empty((nh, H // 8, W // 8, self.mc), dtype=self.dtype, device=self.device)
        for b in range(nh):  # one image at a time: the full-resolution patch matrices of a batch would take gigabytes
            h = ops.nchw_to_nhwc(src[b:b + 1].contiguous(), self.dtype)
            for k, (i, cin, cout, stride) in enumerate(self.hint):
                wt = w[f"hint.{i}.w"]
                cols = ops.im2col3x3(h, stride=stride, ldo=wt.shape[1])
                ho, wo = (h.shape[1] - 1) // stride + 1, (h.shape[2] - 1) // stride + 1
                last = k == len(self.hint) - 1
                h = ops.gemm(cols, wt, w[f"hint.{i}.b"], epilogue=EPI_NONE if last else EPI_SILU,
                             out=out[b].view(ho * wo, cout) if last else None).view(1, ho, wo, cout)
        return out

    # ------------------------------------------------------------------------------------------ forward
    def supports_hint(self, hint: torch.Tensor, n: int, hh: int, ww: int) -> bool:
        """The hint is [1 or n, hint_channels, 8 hh, 8 ww] (what get_control resizes it to, controlnet.py:315-319)."""
        return (hint.dim() == 4 and hint.shape[0] in (1, n) and hint.shape[1] == self.cfg["hint_channels"]
                and hint.shape[2] == 8 * hh and hint.shape[3] == 8 * ww)

    def _zero_conv(self, p: str, h: torch.Tensor, out_dtype: torch.dtype) -> torch.Tensor:
        n, hh, ww, c = h.shape
        z = ops.gemm(h.view(n * hh * ww, c), self.w[p + ".w"], self.w[p + ".b"]).view(n, hh, ww, -1)
        return ops.nhwc_to_nchw(z, out_dtype=out_dtype)

    def forward(self, x: torch.Tensor, hint: torch.Tensor, timesteps: torch.Tensor, context: torch.Tensor,
                y: Optional[torch.Tensor] = None) -> List[torch.Tensor]:
        """cldm.ControlNet.forward (cldm.py:244-270): x NCHW [N,4,h,w] in the compute dtype (already scaled by
        calculate_input), hint [1|N, C_hint, 8h, 8w], timesteps [N], context [N,L,ctx], y [N,adm] -> len(input_blocks) + 1
        fresh contiguous NCHW tensors in x.dtype (Forge scales them in place)."""
        n, _, hh, ww = x.shape
        assert self.supports_hint(hint, n, hh, ww), (tuple(x.shape), tuple(hint.shape))
        gh = self.guided_hint(hint)
        w = self.w
        xn = ops.nchw_to_nhwc(x.to(self.dtype).contiguous(), self.dtype)
        cols = ops.im2col3x3(xn, ldo=64)
        ctx = context.to(self.dtype).contiguous()
        assert ctx.shape[0] == n
        n_ctx = ctx.shape[1]
        ctx2d = ctx.view(n * n_ctx, ctx.shape[2])
        temb_all = self._embeddings(timesteps.float().contiguous(), None if y is None else y.to(self.dtype).contiguous())
        p0 = self.st["input"][0][0][1]
        h = ops.gemm(cols, w[p0 + ".w"], w[p0 + ".b"]).view(n, hh, ww, self.mc)
        ops.add_control_(h, gh, nhwc=True)
        outs = [self._zero_conv(self.zero_convs[0], h, x.dtype)]
        for i, layers in enumerate(self.st["input"][1:], 1):
            h = self._run(layers, h, None, temb_all, ctx2d, n_ctx)
            outs.append(self._zero_conv(self.zero_convs[i], h, x.dtype))
        h = self._run(self.st["middle"], h, None, temb_all, ctx2d, n_ctx)
        outs.append(self._zero_conv(self.zero_convs[-1], h, x.dtype))
        return outs
