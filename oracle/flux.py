"""ORACLE — test infrastructure only (see oracle/ops.py header).

Functional restatement of the reference's Flux transformer forward (backend/nn/flux.py:326-422) over a plain
state dict that uses the reference's own parameter names (`double_blocks.0.img_attn.qkv.weight`, ...).
Arithmetic runs in the dtype of the tensors passed in (fp32 for the oracle); RoPE tables are built in fp64 and
applied in fp32 exactly as the reference does (flux.py:21-49).

Pinned by tests/golden/flux_tiny.pt, generated from the imported reference module by oracle/gen_golden.py.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch

from . import ops as O

SD = Dict[str, torch.Tensor]

# Flux.1-dev as loaded by Forge (huggingface_guess `Flux` unet_config; parameter count 11.90 B, SURVEY.md §8c)
FLUX_DEV = dict(in_channels=16, vec_in_dim=768, context_in_dim=4096, hidden_size=3072, mlp_ratio=4.0, num_heads=24,
                depth=19, depth_single_blocks=38, axes_dim=[16, 56, 56], theta=10000, qkv_bias=True, guidance_embed=True)
# same topology, head dim 128 (the fused path's), two heads, two + two blocks
TINY_FLUX = dict(in_channels=16, vec_in_dim=32, context_in_dim=64, hidden_size=256, mlp_ratio=4.0, num_heads=2,
                 depth=2, depth_single_blocks=2, axes_dim=[16, 56, 56], theta=10000, qkv_bias=True, guidance_embed=True)
CONFIGS = {"flux_dev": FLUX_DEV, "tiny_flux": TINY_FLUX}


def gelu_tanh(x: torch.Tensor) -> torch.Tensor:
    """nn.GELU(approximate="tanh") (flux.py:193,202,280)."""
    return 0.5 * x * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x * x * x)))


def timestep_embedding(t: torch.Tensor, dim: int, max_period: float = 10000.0, time_factor: float = 1000.0):
    """flux.py:52-72: t*1000, fp32 freqs on the device, [cos | sin], cast back to t's dtype."""
    half = dim // 2
    freqs = torch.exp(-math.log(max_period) * torch.arange(half, dtype=torch.float32, device=t.device) / half)
    args = (time_factor * t)[:, None].float() * freqs[None]
    return torch.cat([torch.cos(args), torch.sin(args)], dim=-1).to(t.dtype)


def rope_tables(ids: torch.Tensor, axes_dim, theta: float):
    """flux.py:21-42 + EmbedND (75-89): per position and rotation pair, (cos, sin) in fp32 computed from fp64.
    ids [L, n_axes] -> cos, sin [L, sum(axes_dim)/2]."""
    cs, sn = [], []
    for i, d in enumerate(axes_dim):
        scale = torch.arange(0, d, 2, dtype=torch.float64) / d
        omega = 1.0 / (theta ** scale)
        out = ids[:, i].double().unsqueeze(-1) * omega.unsqueeze(0)
        cs.append(torch.cos(out).float())
        sn.append(torch.sin(out).float())
    return torch.cat(cs, dim=-1), torch.cat(sn, dim=-1)


def apply_rope(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
    """flux.py:45-51 on x [B, H, L, D]: pairs are adjacent elements; out = [[cos, -sin], [sin, cos]] @ (x0, x1),
    computed in fp32 and cast back."""
    xf = x.float().reshape(*x.shape[:-1], -1, 2)
    x0, x1 = xf[..., 0], xf[..., 1]
    o0 = cos * x0 - sin * x1
    o1 = sin * x0 + cos * x1
    return torch.stack([o0, o1], dim=-1).reshape(x.shape).to(x.dtype)


def rms_norm(x: torch.Tensor, scale: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    """RMSNorm (flux.py:115-126) = torch.rms_norm over the last dim."""
    n = torch.rsqrt(torch.mean(x.float() ** 2, dim=-1, keepdim=True) + eps)
    return (x.float() * n).to(x.dtype) * scale.to(x.dtype)


def _mlp_embedder(sd: SD, p: str, x: torch.Tensor) -> torch.Tensor:
    return O.linear(O.silu(O.linear(x, sd[p + ".in_layer.weight"], sd[p + ".in_layer.bias"])),
                    sd[p + ".out_layer.weight"], sd[p + ".out_layer.bias"])


def _modulation(sd: SD, p: str, vec: torch.Tensor, n: int):
    out = O.linear(O.silu(vec), sd[p + ".lin.weight"], sd[p + ".lin.bias"])[:, None, :]
    return out.chunk(n, dim=-1)


def _ln(x):
    return O.layer_norm(x, None, None, 1e-6)


def _split_heads(qkv: torch.Tensor, H: int):
    B, L, _ = qkv.shape
    q, k, v = qkv.view(B, L, 3, H, -1).permute(2, 0, 3, 1, 4)
    return q, k, v


def _attention(q, k, v, cos, sin):
    """flux.py:15-18: rope on q and k, then softmax(q k^T / sqrt(D)) v, heads merged -> [B, L, H*D]."""
    q, k = apply_rope(q, cos, sin), apply_rope(k, cos, sin)
    B, H, L, D = q.shape
    s = torch.matmul(q.float(), k.float().transpose(-1, -2)) * (D ** -0.5)
    o = torch.matmul(torch.softmax(s, dim=-1), v.float()).to(q.dtype)
    return o.permute(0, 2, 1, 3).reshape(B, L, H * D)


def double_block(sd: SD, p: str, H: int, img, txt, vec, cos, sin):
    """DoubleStreamBlock.forward (flux.py:206-264)."""
    i_s1, i_c1, i_g1, i_s2, i_c2, i_g2 = _modulation(sd, p + ".img_mod", vec, 6)
    t_s1, t_c1, t_g1, t_s2, t_c2, t_g2 = _modulation(sd, p + ".txt_mod", vec, 6)
    iq, ik, iv = _split_heads(O.linear((1 + i_c1) * _ln(img) + i_s1, sd[p + ".img_attn.qkv.weight"], sd.get(p + ".img_attn.qkv.bias")), H)
    iq, ik = rms_norm(iq, sd[p + ".img_attn.norm.query_norm.scale"]), rms_norm(ik, sd[p + ".img_attn.norm.key_norm.scale"])
    tq, tk, tv = _split_heads(O.linear((1 + t_c1) * _ln(txt) + t_s1, sd[p + ".txt_attn.qkv.weight"], sd.get(p + ".txt_attn.qkv.bias")), H)
    tq, tk = rms_norm(tq, sd[p + ".txt_attn.norm.query_norm.scale"]), rms_norm(tk, sd[p + ".txt_attn.norm.key_norm.scale"])
    attn = _attention(torch.cat((tq, iq), 2), torch.cat((tk, ik), 2), torch.cat((tv, iv), 2), cos, sin)
    Lt = txt.shape[1]
    t_attn, i_attn = attn[:, :Lt], attn[:, Lt:]

    def mlp(q, x):
        return O.linear(gelu_tanh(O.linear(x, sd[q + ".0.weight"], sd[q + ".0.bias"])), sd[q + ".2.weight"], sd[q + ".2.bias"])

    img = img + i_g1 * O.linear(i_attn, sd[p + ".img_attn.proj.weight"], sd[p + ".img_attn.proj.bias"])
    img = img + i_g2 * mlp(p + ".img_mlp", (1 + i_c2) * _ln(img) + i_s2)
    txt = txt + t_g1 * O.linear(t_attn, sd[p + ".txt_attn.proj.weight"], sd[p + ".txt_attn.proj.bias"])
    txt = txt + t_g2 * mlp(p + ".txt_mlp", (1 + t_c2) * _ln(txt) + t_s2)
    return img, txt  # fp16_fix (backend/utils.py:104-111) is the identity outside fp16


def single_block(sd: SD, p: str, H: int, hidden: int, x, vec, cos, sin):
    """SingleStreamBlock.forward (flux.py:283-307)."""
    shift, scale, gate = _modulation(sd, p + ".modulation", vec, 3)
    y = O.linear((1 + scale) * _ln(x) + shift, sd[p + ".linear1.weight"], sd[p + ".linear1.bias"])
    qkv, mlp = y[..., :3 * hidden], y[..., 3 * hidden:]
    q, k, v = _split_heads(qkv, H)
    q, k = rms_norm(q, sd[p + ".norm.query_norm.scale"]), rms_norm(k, sd[p + ".norm.key_norm.scale"])
    attn = _attention(q, k, v, cos, sin)
    out = O.linear(torch.cat((attn, gelu_tanh(mlp)), 2), sd[p + ".linear2.weight"], sd[p + ".linear2.bias"])
    return x + gate * out


def position_ids(h_len: int, w_len: int, txt_len: int) -> torch.Tensor:
    """flux.py:402-409: txt ids all zero, img ids (0, row, col); concatenated txt first (flux.py:363)."""
    img = torch.zeros(h_len, w_len, 3)
    img[..., 1] += torch.arange(h_len, dtype=torch.float32)[:, None]
    img[..., 2] += torch.arange(w_len, dtype=torch.float32)[None, :]
    return torch.cat([torch.zeros(txt_len, 3), img.reshape(-1, 3)], dim=0)


def patchify(x: torch.Tensor) -> torch.Tensor:
    """flux.py:398-399 (even h, w: the circular pad is empty): b c (h 2) (w 2) -> b (h w) (c 2 2)."""
    B, C, Hh, Ww = x.shape
    return x.view(B, C, Hh // 2, 2, Ww // 2, 2).permute(0, 2, 4, 1, 3, 5).reshape(B, (Hh // 2) * (Ww // 2), C * 4)


def unpatchify(o: torch.Tensor, C: int, Hh: int, Ww: int) -> torch.Tensor:
    """flux.py:412."""
    B = o.shape[0]
    return o.view(B, Hh // 2, Ww // 2, C, 2, 2).permute(0, 3, 1, 4, 2, 5).reshape(B, C, Hh, Ww)


def flux_forward(sd: SD, cfg: dict, x: torch.Tensor, timestep: torch.Tensor, context: torch.Tensor, y: torch.Tensor,
                 guidance: Optional[torch.Tensor] = None) -> torch.Tensor:
    """IntegratedFluxTransformer2DModel.forward (flux.py:389-422); odd latent sizes are padded circularly to the patch size
    (:394-397) and the output is cropped back (:412)."""
    h0, w0 = x.shape[2], x.shape[3]
    if (h0 | w0) & 1:
        xp = torch.nn.functional.pad(x, (0, w0 & 1, 0, h0 & 1), mode="circular")
        return flux_forward(sd, cfg, xp, timestep, context, y, guidance)[:, :, :h0, :w0]
    B, C, Hh, Ww = x.shape
    H, hidden = cfg["num_heads"], cfg["hidden_size"]
    img = O.linear(patchify(x), sd["img_in.weight"], sd["img_in.bias"])
    vec = _mlp_embedder(sd, "time_in", timestep_embedding(timestep, 256).to(img.dtype))
    if cfg["guidance_embed"]:
        vec = vec + _mlp_embedder(sd, "guidance_in", timestep_embedding(guidance, 256).to(img.dtype))
    vec = vec + _mlp_embedder(sd, "vector_in", y)
    txt = O.linear(context, sd["txt_in.weight"], sd["txt_in.bias"])
    Lt = txt.shape[1]
    cos, sin = rope_tables(position_ids(Hh // 2, Ww // 2, Lt), cfg["axes_dim"], cfg["theta"])
    cos, sin = cos.to(x.device), sin.to(x.device)
    for i in range(cfg["depth"]):
        img, txt = double_block(sd, f"double_blocks.{i}", H, img, txt, vec, cos, sin)
    xx = torch.cat((txt, img), 1)
    for i in range(cfg["depth_single_blocks"]):
        xx = single_block(sd, f"single_blocks.{i}", H, hidden, xx, vec, cos, sin)
    img = xx[:, Lt:]
    shift, scale = O.linear(O.silu(vec), sd["final_layer.adaLN_modulation.1.weight"], sd["final_layer.adaLN_modulation.1.bias"]).chunk(2, dim=1)
    img = (1 + scale[:, None, :]) * _ln(img) + shift[:, None, :]
    out = O.linear(img, sd["final_layer.linear.weight"], sd["final_layer.linear.bias"])
    return unpatchify(out, C, Hh, Ww)


def random_state_dict(cfg: dict, seed: int = 0, dtype=torch.float32, device=None) -> SD:
    """Deterministic synthetic weights with the reference's parameter names and shapes (same conventions as
    oracle.unet.random_state_dict).  Modulation weights are scaled down so (1 + scale) stays near 1 and gates near
    0.3: the residual stream keeps O(1) magnitude through all blocks."""
    g = torch.Generator().manual_seed(seed)
    assert device in (None, "cpu", "meta"), device

    def randn(*shape):  # device="meta": names and shapes only, nothing drawn or allocated
        return torch.empty(*shape, device="meta") if device == "meta" else torch.randn(*shape, generator=g)

    sd: SD = {}

    def lin(p, cin, cout, bias=True, wscale=1.0, bmean=0.0):
        sd[p + ".weight"] = (randn(cout, cin) * (wscale * cin ** -0.5)).to(dtype)
        if bias:
            sd[p + ".bias"] = (bmean + randn(cout) * 0.05).to(dtype)

    hs, H = cfg["hidden_size"], cfg["num_heads"]
    D = hs // H
    mlp = int(hs * cfg["mlp_ratio"])
    lin("img_in", cfg["in_channels"] * 4, hs)
    for name, cin in (("time_in", 256), ("vector_in", cfg["vec_in_dim"])) + ((("guidance_in", 256),) if cfg["guidance_embed"] else ()):
        lin(name + ".in_layer", cin, hs)
        lin(name + ".out_layer", hs, hs)
    lin("txt_in", cfg["context_in_dim"], hs)

    def qknorm(p):
        sd[p + ".query_norm.scale"] = (1.0 + 0.1 * randn(D)).to(dtype)
        sd[p + ".key_norm.scale"] = (1.0 + 0.1 * randn(D)).to(dtype)

    for i in range(cfg["depth"]):
        p = f"double_blocks.{i}"
        for s in ("img", "txt"):
            lin(f"{p}.{s}_mod.lin", hs, 6 * hs, wscale=0.3, bmean=0.1)
            lin(f"{p}.{s}_attn.qkv", hs, 3 * hs, bias=cfg["qkv_bias"])
            qknorm(f"{p}.{s}_attn.norm")
            lin(f"{p}.{s}_attn.proj", hs, hs)
            lin(f"{p}.{s}_mlp.0", hs, mlp)
            lin(f"{p}.{s}_mlp.2", mlp, hs)
    for i in range(cfg["depth_single_blocks"]):
        p = f"single_blocks.{i}"
        lin(p + ".linear1", hs, 3 * hs + mlp)
        lin(p + ".linear2", hs + mlp, hs)
        qknorm(p + ".norm")
        lin(p + ".modulation.lin", hs, 3 * hs, wscale=0.3, bmean=0.1)
    lin("final_layer.linear", hs, 4 * cfg["in_channels"])
    lin("final_layer.adaLN_modulation.1", hs, 2 * hs, wscale=0.3)
    return sd
