"""ORACLE — test infrastructure only (see oracle/ops.py header).

Functional restatement of the reference's LDM UNet forward (backend/nn/unet.py) over a plain state dict
that uses the reference's own parameter names (`input_blocks.1.0.in_layers.2.weight`, ...).  The plain
txt2img path only: no control, no patches, no block modifiers (the fast-path predicate of SURVEY.md §8b).
Arithmetic runs in the dtype of the tensors passed in (fp32 for the oracle; the reference's fp16 GPU run
rounds to fp16 after every op, which is the tolerance the parity tests state).
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import ops as O

SD = Dict[str, torch.Tensor]


def structure(cfg: dict):
    """Replays the constructor of IntegratedUNet2DConditionModel (backend/nn/unet.py:481-693) and returns
    the block lists as tuples:
      ("conv", prefix, cin, cout) | ("res", prefix, cin, cout) | ("attn", prefix, ch, heads, dim_head, depth)
      | ("down", prefix, ch) | ("up", prefix, ch)
    """
    mc = cfg["model_channels"]
    nrb = cfg["num_res_blocks"]
    cm = cfg["channel_mult"]
    if isinstance(nrb, int):
        nrb = len(cm) * [nrb]
    td = list(cfg["transformer_depth"])
    tdo = list(cfg["transformer_depth_output"])
    nh, nhc = cfg["num_heads"], cfg["num_head_channels"]

    def heads_of(ch):
        if nhc == -1:
            return nh, ch // nh
        return ch // nhc, nhc

    input_blocks: List[list] = [[("conv", "input_blocks.0.0", cfg["in_channels"], mc)]]
    chans = [mc]
    ch = mc
    idx = 1
    for level, mult in enumerate(cm):
        for _ in range(nrb[level]):
            layers = [("res", f"input_blocks.{idx}.0", ch, mult * mc)]
            ch = mult * mc
            depth = td.pop(0)
            if depth > 0:
                h, dh = heads_of(ch)
                layers.append(("attn", f"input_blocks.{idx}.1", ch, h, dh, depth))
            input_blocks.append(layers)
            chans.append(ch)
            idx += 1
        if level != len(cm) - 1:
            input_blocks.append([("down", f"input_blocks.{idx}.0", ch)])
            chans.append(ch)
            idx += 1
    h, dh = heads_of(ch)
    middle = [("res", "middle_block.0", ch, ch)]
    if cfg["transformer_depth_middle"] >= 0:
        middle += [("attn", "middle_block.1", ch, h, dh, cfg["transformer_depth_middle"]),
                   ("res", "middle_block.2", ch, ch)]
    output_blocks: List[list] = []
    idx = 0
    for level, mult in list(enumerate(cm))[::-1]:
        for i in range(nrb[level] + 1):
            ich = chans.pop()
            layers = [("res", f"output_blocks.{idx}.0", ch + ich, mc * mult)]
            ch = mc * mult
            depth = tdo.pop()
            j = 1
            if depth > 0:
                h, dh = heads_of(ch)
                layers.append(("attn", f"output_blocks.{idx}.{j}", ch, h, dh, depth))
                j += 1
            if level and i == nrb[level]:
                layers.append(("up", f"output_blocks.{idx}.{j}", ch))
            output_blocks.append(layers)
            idx += 1
    return dict(input=input_blocks, middle=middle, output=output_blocks, out_ch=ch)


def _lin(sd: SD, p: str, x):
    return O.linear(x, sd[p + ".weight"], sd.get(p + ".bias"))


def _conv(sd: SD, p: str, x, stride=1, padding=1):
    return O.conv2d(x, sd[p + ".weight"], sd.get(p + ".bias"), stride=stride, padding=padding)


def _gn(sd: SD, p: str, x, eps):
    return O.group_norm(x, 32, sd[p + ".weight"], sd[p + ".bias"], eps)


def _ln(sd: SD, p: str, x):
    return O.layer_norm(x, sd[p + ".weight"], sd[p + ".bias"], 1e-5)


def res_block(sd: SD, p: str, x, emb):
    """backend/nn/unet.py:433-478 (ResBlock._forward; updown=False, use_scale_shift_norm=False)."""
    h = _conv(sd, p + ".in_layers.2", O.silu(_gn(sd, p + ".in_layers.0", x, 1e-5)))
    emb_out = _lin(sd, p + ".emb_layers.1", O.silu(emb)).type(h.dtype)
    h = h + emb_out[..., None, None]
    h = _conv(sd, p + ".out_layers.3", O.silu(_gn(sd, p + ".out_layers.0", h, 1e-5)))
    if (p + ".skip_connection.weight") in sd:
        x = _conv(sd, p + ".skip_connection", x, padding=0)
    return x + h


def cross_attention(sd: SD, p: str, x, context, heads):
    """backend/nn/unet.py:145-155 (CrossAttention.forward)."""
    q = _lin(sd, p + ".to_q", x)
    context = x if context is None else context
    k = _lin(sd, p + ".to_k", context)
    v = _lin(sd, p + ".to_v", context)
    out = O.attention(q, k, v, heads)
    return _lin(sd, p + ".to_out.0", out)


def transformer_block(sd: SD, p: str, x, context, heads):
    """backend/nn/unet.py:183-279 (BasicTransformerBlock._forward, no patches, ff_in off, is_res)."""
    x = x + cross_attention(sd, p + ".attn1", _ln(sd, p + ".norm1", x), None, heads)
    x = x + cross_attention(sd, p + ".attn2", _ln(sd, p + ".norm2", x), context, heads)
    n = _ln(sd, p + ".norm3", x)
    ff = O.geglu(n, sd[p + ".ff.net.0.proj.weight"], sd[p + ".ff.net.0.proj.bias"])
    ff = _lin(sd, p + ".ff.net.2", ff)
    return x + ff


def spatial_transformer(sd: SD, p: str, x, context, heads, depth, use_linear):
    """backend/nn/unet.py:308-327 (SpatialTransformer.forward)."""
    b, c, hh, ww = x.shape
    x_in = x
    x = _gn(sd, p + ".norm", x, 1e-6)
    if not use_linear:
        x = _conv(sd, p + ".proj_in", x, padding=0)
    x = x.permute(0, 2, 3, 1).reshape(b, hh * ww, -1)
    if use_linear:
        x = _lin(sd, p + ".proj_in", x)
    for d in range(depth):
        x = transformer_block(sd, f"{p}.transformer_blocks.{d}", x, context, heads)
    if use_linear:
        x = _lin(sd, p + ".proj_out", x)
    x = x.reshape(b, hh, ww, -1).permute(0, 3, 1, 2)
    if not use_linear:
        x = _conv(sd, p + ".proj_out", x, padding=0)
    return x + x_in


def _run_layers(sd: SD, cfg: dict, layers, h, emb, context):
    for layer in layers:
        kind, p = layer[0], layer[1]
        if kind == "conv":
            h = _conv(sd, p, h)
        elif kind == "res":
            h = res_block(sd, p, h, emb)
        elif kind == "attn":
            h = spatial_transformer(sd, p, h, context, layer[3], layer[5], cfg["use_linear_in_transformer"])
        elif kind == "down":
            h = _conv(sd, p + ".op", h, stride=2)  # backend/nn/unet.py:358-374
        elif kind == "up":
            h = _conv(sd, p + ".conv", O.upsample_nearest2x(h))  # backend/nn/unet.py:330-355
    return h


def _apply_control(h, control, name):
    """backend/nn/unet.py:44-52."""
    if control is not None and name in control and len(control[name]) > 0:
        ctrl = control[name].pop()
        if ctrl is not None:
            h = h + ctrl
    return h


def unet_forward(sd: SD, cfg: dict, x, timesteps, context, y: Optional[torch.Tensor] = None, control: Optional[dict] = None):
    """backend/nn/unet.py:696-763 (IntegratedUNet2DConditionModel.forward, plain path; `control` = ControlNet residual
    lists consumed from their ends, :714, 733, 739)."""
    if control is not None:
        control = {k: list(v) for k, v in control.items()}
    st = structure(cfg)
    t_emb = O.timestep_embedding(timesteps, cfg["model_channels"]).to(x.dtype)
    emb = _lin(sd, "time_embed.2", O.silu(_lin(sd, "time_embed.0", t_emb)))
    if cfg.get("num_classes") is not None:
        assert y is not None and cfg["num_classes"] == "sequential"
        emb = emb + _lin(sd, "label_emb.0.2", O.silu(_lin(sd, "label_emb.0.0", y)))
    hs = []
    h = x
    for layers in st["input"]:
        h = _apply_control(_run_layers(sd, cfg, layers, h, emb, context), control, "input")
        hs.append(h)
    h = _apply_control(_run_layers(sd, cfg, st["middle"], h, emb, context), control, "middle")
    for layers in st["output"]:
        h = torch.cat([h, _apply_control(hs.pop(), control, "output")], dim=1)
        h = _run_layers(sd, cfg, layers, h, emb, context)
    h = _conv(sd, "out.2", O.silu(_gn(sd, "out.0", h, 1e-5)))
    return h.type(x.dtype)


def random_state_dict(cfg: dict, seed: int = 0, dtype=torch.float32, device=None) -> SD:
    """Deterministic synthetic weights with the reference's parameter names and shapes.
    ForgeOperations.*.reset_parameters are no-ops (backend/operations.py:166-167), so there is no reference
    initialisation to mirror; weights are N(0, 1/fan_in)-scaled so activations stay O(1) through the net,
    norm gains ~ 1, biases small."""
    g = torch.Generator().manual_seed(seed)
    assert device in (None, "cpu", "meta"), device

    def randn(*shape):  # device="meta": names and shapes only, nothing drawn or allocated
        return torch.empty(*shape, device="meta") if device == "meta" else torch.randn(*shape, generator=g)

    sd: SD = {}

    def lin(p, cin, cout, bias=True):
        sd[p + ".weight"] = (randn(cout, cin) * cin ** -0.5).to(dtype)
        if bias:
            sd[p + ".bias"] = (randn(cout) * 0.05).to(dtype)

    def conv(p, cin, cout, k):
        sd[p + ".weight"] = (randn(cout, cin, k, k) * (cin * k * k) ** -0.5).to(dtype)
        sd[p + ".bias"] = (randn(cout) * 0.05).to(dtype)

    def norm(p, c):
        sd[p + ".weight"] = (1.0 + 0.1 * randn(c)).to(dtype)
        sd[p + ".bias"] = (0.05 * randn(c)).to(dtype)

    mc = cfg["model_channels"]
    ted = mc * 4
    lin("time_embed.0", mc, ted)
    lin("time_embed.2", ted, ted)
    if cfg.get("num_classes") == "sequential":
        lin("label_emb.0.0", cfg["adm_in_channels"], ted)
        lin("label_emb.0.2", ted, ted)
    st = structure(cfg)
    ctx = cfg["context_dim"]
    use_lin = cfg["use_linear_in_transformer"]

    def add(layer):
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
            ch, depth = layer[2], layer[5]
            norm(p + ".norm", ch)
            if use_lin:
                lin(p + ".proj_in", ch, ch)
                lin(p + ".proj_out", ch, ch)
            else:
                conv(p + ".proj_in", ch, ch, 1)
                conv(p + ".proj_out", ch, ch, 1)
            for d in range(depth):
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
        elif kind == "up":
            conv(p + ".conv", layer[2], layer[2], 3)

    for blk in st["input"] + [st["middle"]] + st["output"]:
        for layer in blk:
            add(layer)
    norm("out.0", st["out_ch"])
    conv("out.2", mc, cfg["out_channels"], 3)
    return sd
