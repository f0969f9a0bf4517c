"""ORACLE — test infrastructure only (see oracle/ops.py header).

Functional restatement of the reference's ControlNet forward (backend/nn/cnets/cldm.py:244-270) over a plain state dict
with the reference's own parameter names, built on oracle/unet.py's block functions, plus the ControlNet configurations
and seeded synthetic weights the tests use.  The configurations live here rather than in oracle/configs.py, and the golden
generator in oracle/gen_controlnet_golden.py rather than in oracle/gen_golden.py, so that the oracle modules the existing
tests and fixtures are pinned to stay exactly as they were.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import configs as CF
from . import ops as O
from . import unet as OU

SD = Dict[str, torch.Tensor]

_ENCODER_KEYS = ("in_channels", "model_channels", "num_res_blocks", "channel_mult", "transformer_depth",
                 "transformer_depth_middle", "num_heads", "num_head_channels", "use_spatial_transformer",
                 "use_linear_in_transformer", "context_dim", "adm_in_channels", "num_classes")


def controlnet_of(unet_cfg: dict, hint_channels: int = 3) -> dict:
    """The ControlNet of a UNet configuration: its encoder half (cldm.ControlNet's constructor arguments) + hint channels."""
    return dict({k: unet_cfg[k] for k in _ENCODER_KEYS}, hint_channels=hint_channels)


# full-size diffusers SDXL ControlNet in LDM form (the SDXL encoder: transformer depths [0,0,2,2,10,10], middle 10)
SDXL_CONTROLNET = controlnet_of(CF.SDXL)
SD15_CONTROLNET = controlnet_of(CF.SD15)
TINY_XL_CONTROLNET = controlnet_of(CF.TINY_XL)
TINY_15H_CONTROLNET = controlnet_of(CF.TINY_15H)   # head dims 8/16/32: the head-dim padding of the fused path
# no cross-attention anywhere (as in some small SDXL ControlNets): a depth-0 SpatialTransformer in the middle block, or none
TINY_XL_NOATTN = dict(TINY_XL_CONTROLNET, transformer_depth=[0] * 6, transformer_depth_middle=0)
TINY_XL_NOATTN_NOMID = dict(TINY_XL_NOATTN, transformer_depth_middle=-1)
CONFIGS = {"sdxl": SDXL_CONTROLNET, "sd15": SD15_CONTROLNET, "tiny_xl": TINY_XL_CONTROLNET, "tiny_15h": TINY_15H_CONTROLNET,
           "tiny_xl_noattn": TINY_XL_NOATTN, "tiny_xl_noattn_nomid": TINY_XL_NOATTN_NOMID}


def hint_layers(cfg: dict):
    """(index in input_hint_block, Cin, Cout, stride) of its eight convolutions (cldm.py:116-132)."""
    ch = [cfg["hint_channels"], 16, 16, 32, 32, 96, 96, 256, cfg["model_channels"]]
    st = [1, 1, 2, 1, 2, 1, 2, 1]
    return [(2 * i, ch[i], ch[i + 1], st[i]) for i in range(8)]


def structure(cfg: dict):
    """Input blocks and middle block of cldm.ControlNet (its constructor order is the UNet encoder's)."""
    nrb = cfg["num_res_blocks"]
    n_out = (len(cfg["channel_mult"]) * nrb if isinstance(nrb, int) else sum(nrb)) + len(cfg["channel_mult"])
    st = OU.structure(dict(cfg, transformer_depth_output=[0] * n_out))  # the decoder half is built and dropped
    return st["input"], st["middle"]


def hint_block(sd: SD, cfg: dict, hint, dtype) -> torch.Tensor:
    """input_hint_block (cldm.py:116-132): eight 3x3 convolutions with SiLU between them, hint -> latent resolution."""
    g = hint.to(dtype)
    layers = hint_layers(cfg)
    for k, (i, _, _, stride) in enumerate(layers):
        g = OU._conv(sd, f"input_hint_block.{i}", g, stride=stride)
        if k + 1 < len(layers):
            g = O.silu(g)
    return g


def controlnet_forward(sd: SD, cfg: dict, x, hint, timesteps, context, y: Optional[torch.Tensor] = None,
                       guided_hint: Optional[torch.Tensor] = None) -> List[torch.Tensor]:
    """cldm.ControlNet.forward: len(input_blocks) + 1 residuals, the hint encoder's output (batch 1 or N) added after
    the first input block.  `guided_hint`: hint_block(hint) computed beforehand (the reference recomputes it per call)."""
    inp, mid = structure(cfg)
    t_emb = O.timestep_embedding(timesteps, cfg["model_channels"]).to(x.dtype)
    emb = OU._lin(sd, "time_embed.2", O.silu(OU._lin(sd, "time_embed.0", t_emb)))
    g = hint_block(sd, cfg, hint, x.dtype) if guided_hint is None else guided_hint
    if cfg.get("num_classes") is not None:
        emb = emb + OU._lin(sd, "label_emb.0.2", O.silu(OU._lin(sd, "label_emb.0.0", y)))
    outs = []
    h = x
    for i, blk in enumerate(inp):
        h = OU._run_layers(sd, cfg, blk, h, emb, context)
        if i == 0:
            h = h + g
        outs.append(OU._conv(sd, f"zero_convs.{i}.0", h, padding=0))
    h = OU._run_layers(sd, cfg, mid, h, emb, context)
    outs.append(OU._conv(sd, "middle_block_out.0", h, padding=0))
    return outs


def random_controlnet_state_dict(cfg: dict, hint_channels: int = 3, seed: int = 0, dtype=torch.float32) -> SD:
    """Seeded synthetic weights under the reference's names.  The zero convs get non-zero weights (a trained ControlNet's
    are no longer zero), so that every output depends on the whole network."""
    cfg = dict(cfg, hint_channels=hint_channels)
    g = torch.Generator().manual_seed(seed)
    randn = lambda *s: torch.randn(*s, generator=g)  # noqa: E731
    sd: SD = {}

    def lin(p, cin, cout, bias=True):
        sd[p + ".weight"] = (randn(cout, cin) * cin ** -0.5).to(dtype)
        if bias:
            sd[p + ".bias"] = (randn(cout) * 0.05).to(dtype)

    def conv(p, cin, cout, k, gain=1.0):
        sd[p + ".weight"] = (randn(cout, cin, k, k) * gain * (cin * k * k) ** -0.5).to(dtype)
        sd[p + ".bias"] = (randn(cout) * 0.05).to(dtype)

    def norm(p, c):
        sd[p + ".weight"] = (1.0 + 0.1 * randn(c)).to(dtype)
        sd[p + ".bias"] = (0.05 * randn(c)).to(dtype)

    mc, ted, ctx = cfg["model_channels"], 4 * cfg["model_channels"], cfg["context_dim"]
    lin("time_embed.0", mc, ted)
    lin("time_embed.2", ted, ted)
    if cfg.get("num_classes") == "sequential":
        lin("label_emb.0.0", cfg["adm_in_channels"], ted)
        lin("label_emb.0.2", ted, ted)
    for i, cin, cout, _ in hint_layers(cfg):
        conv(f"input_hint_block.{i}", cin, cout, 3, gain=1.5)  # SiLU halves the scale: keep the hint features O(1)
    inp, mid = structure(cfg)
    for layer in [ly for blk in inp for ly in blk] + mid:
        kind, p = layer[0], layer[1]
        if kind == "conv":
            conv(p, layer[2], layer[3], 3)
        elif kind == "res":
            cin, cout = layer[2], layer[3]
            norm(p + ".in_layers.0", cin)
            conv(p + ".in_layers.2", cin, cout, 3)
            lin(p + ".emb_layers.1", ted, cout)
            norm(p + ".out_layers.0", cout)
            conv(p + ".out_layers.3", cout, cout, 3)
            if cin != cout:
                conv(p + ".skip_connection", cin, cout, 1)
        elif kind == "attn":
            ch = layer[2]
            norm(p + ".norm", ch)
            for n in ("proj_in", "proj_out"):
                if cfg["use_linear_in_transformer"]:
                    lin(f"{p}.{n}", ch, ch)
                else:
                    conv(f"{p}.{n}", ch, ch, 1)
            for d in range(layer[5]):
                q = f"{p}.transformer_blocks.{d}"
                for a, kv in (("attn1", ch), ("attn2", ctx)):
                    lin(f"{q}.{a}.to_q", ch, ch, bias=False)
                    lin(f"{q}.{a}.to_k", kv, ch, bias=False)
                    lin(f"{q}.{a}.to_v", kv, ch, bias=False)
                    lin(f"{q}.{a}.to_out.0", ch, ch)
                for n in ("norm1", "norm2", "norm3"):
                    norm(f"{q}.{n}", ch)
                lin(f"{q}.ff.net.0.proj", ch, ch * 8)
                lin(f"{q}.ff.net.2", ch * 4, ch)
        elif kind == "down":
            conv(p + ".op", layer[2], layer[2], 3)
    chans = [blk[0][3] if blk[0][0] in ("conv", "res") else blk[0][2] for blk in inp]
    for i, c in enumerate(chans):
        conv(f"zero_convs.{i}.0", c, c, 1)
    conv("middle_block_out.0", chans[-1], chans[-1], 1)
    return sd
