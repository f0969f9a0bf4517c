"""Fused channels-last UNet forward for the LDM UNet of SD1.x / SDXL — the B200 replacement for
`IntegratedUNet2DConditionModel.forward` (reference backend/nn/unet.py:696-763) on the plain txt2img path
(no control / patches / block modifiers: the fast-path predicate of SURVEY.md §8b).

The engine consumes a state dict with the reference's own parameter names, repacks the weights once
(3x3 filters -> [Cout, 9*Cin], fused QKV / KV projections, GEGLU row interleave, all ResBlock
time-embedding projections stacked into one matrix) and then runs the forward as a flat sequence of
libb200forge launches on NHWC activations:

  ResBlock            GN-stats -> GN-apply+SiLU(+concat) -> conv3x3(+bias +temb) -> GN -> conv3x3(+bias +skip)
  SpatialTransformer  GN -> proj_in GEMM -> depth x [QKV GEMM(LN1 folded) -> attention -> out GEMM(+res, row stats)
                                                      Q GEMM(LN2 folded), K|V from the per-job cache -> attention
                                                                                          -> out GEMM(+res, row stats)
                                                      GEGLU GEMM(LN3 folded) -> FF-out GEMM(+res, row stats)]
                      -> proj_out GEMM(+res)
  LayerNorm           never a kernel: gamma is folded into the consumer GEMM's weights, mean / rstd are applied in its
                      epilogue from row sums that the producer GEMM's epilogue accumulated (ops.fold_layernorm)
  cross-attention K|V projected once per job from the constant context (fill_kv_cache), not once per step
  head dims           40 / 80 (SD1.5) zero-padded to 64 / 128 in the packed projections; 160 through one
                      GEMM -> block-diagonal softmax -> GEMM per head over the whole batch (ops.attention_blockdiag)
  skip concat         never materialised: GN-apply, the 1x1 skip GEMM and the conv read both sources

No torch operator runs on the data path; torch only provides buffers (`torch.empty`) and the stream.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import ops
from .ops import EPI_GEGLU, EPI_NONE, EPI_SILU

SD = Dict[str, torch.Tensor]


def encoder_structure(cfg: dict):
    """Input blocks and middle block of the LDM UNet encoder, shared by the UNet and by cldm.ControlNet, whose constructors
    build them in the same order (backend/nn/unet.py:481-620, backend/nn/cnets/cldm.py:131-234):
    (input, middle, chans, ch) with chans the channel count after every input block and ch the middle block's."""
    mc = cfg["model_channels"]
    nrb = cfg["num_res_blocks"]
    cm = list(cfg["channel_mult"])
    if isinstance(nrb, int):
        nrb = len(cm) * [nrb]
    td = list(cfg["transformer_depth"])
    nh, nhc = cfg["num_heads"], cfg["num_head_channels"]

    def heads_of(ch):
        return (nh, ch // nh) if nhc == -1 else (ch // nhc, nhc)

    inp = [[("conv", "input_blocks.0.0", cfg["in_channels"], mc)]]
    chans = [mc]
    ch = mc
    i = 1
    for level, mult in enumerate(cm):
        for _ in range(nrb[level]):
            layers = [("res", f"input_blocks.{i}.0", ch, mult * mc)]
            ch = mult * mc
            depth = td.pop(0)
            if depth > 0:
                h, dh = heads_of(ch)
                layers.append(("attn", f"input_blocks.{i}.1", ch, h, dh, depth))
            inp.append(layers)
            chans.append(ch)
            i += 1
        if level != len(cm) - 1:
            inp.append([("down", f"input_blocks.{i}.0", ch)])
            chans.append(ch)
            i += 1
    h, dh = heads_of(ch)
    mid = [("res", "middle_block.0", ch, ch)]
    if cfg["transformer_depth_middle"] >= 0:
        mid += [("attn", "middle_block.1", ch, h, dh, cfg["transformer_depth_middle"]),
                ("res", "middle_block.2", ch, ch)]
    return inp, mid, chans, ch


def unet_structure(cfg: dict):
    """Block list of the LDM UNet for a config (mirrors the constructor order of backend/nn/unet.py:481-693):
    ("conv"|"res"|"attn"|"down"|"up", prefix, ...)."""
    mc = cfg["model_channels"]
    nrb = cfg["num_res_blocks"]
    cm = list(cfg["channel_mult"])
    if isinstance(nrb, int):
        nrb = len(cm) * [nrb]
    tdo = list(cfg["transformer_depth_output"])
    nh, nhc = cfg["num_heads"], cfg["num_head_channels"]

    def heads_of(ch):
        return (nh, ch // nh) if nhc == -1 else (ch // nhc, nhc)

    inp, mid, chans, ch = encoder_structure(cfg)
    out = []
    i = 0
    for level, mult in list(enumerate(cm))[::-1]:
        for k in range(nrb[level] + 1):
            ich = chans.pop()
            layers = [("res", f"output_blocks.{i}.0", ch + ich, mc * mult, ch, ich)]
            ch = mc * mult
            depth = tdo.pop()
            j = 1
            if depth > 0:
                h, dh = heads_of(ch)
                layers.append(("attn", f"output_blocks.{i}.{j}", ch, h, dh, depth))
                j += 1
            if level and k == nrb[level]:
                layers.append(("up", f"output_blocks.{i}.{j}", ch))
            out.append(layers)
            i += 1
    return dict(input=inp, middle=mid, output=out, out_ch=ch)


class UNetEngine:
    """Weights packed for the sm_100a kernels + the launch sequence of one forward."""

    def __init__(self, cfg: dict, state_dict: SD, dtype: torch.dtype = torch.float16, device="cuda"):
        self.cfg = dict(cfg)
        self.dtype = dtype
        self.device = torch.device(device)
        self.st = self._structure(cfg)
        self.mc = cfg["model_channels"]
        self.ted = self.mc * 4
        self.has_label = cfg.get("num_classes") is not None
        self.w: Dict[str, torch.Tensor] = {}
        self.head_pad: Dict[str, tuple] = {}
        if self.device.type == "cuda":
            ops.gn_workspace(self.device)  # created (zeroed) here so that it never happens inside a graph capture
        self._pack(state_dict)

    @staticmethod
    def _structure(cfg: dict) -> dict:
        return unet_structure(cfg)

    # ------------------------------------------------------------------------------------------ packing
    def repack(self, state_dict: SD) -> None:
        """Re-pack after the module's parameters changed (Forge merged or removed a LoRA): same buffers, new contents."""
        old, self.w = self.w, {}
        self._pack(state_dict)
        self.w = ops.refresh_packed(old, self.w)

    def _t(self, t: torch.Tensor) -> torch.Tensor:
        return t.detach().to(device=self.device, dtype=self.dtype).contiguous()

    def _pack(self, sd: SD) -> None:
        w = self.w
        g = lambda k: self._t(sd[k])  # noqa: E731
        self._pack_embeddings(g)
        self._pack_blocks(g, self.st["input"] + [self.st["middle"]] + self.st["output"])
        w["out.0.g"], w["out.0.b"] = g("out.0.weight"), g("out.0.bias")
        ow = ops.pack_conv3x3(g("out.2.weight"))  # [4, 9*mc] -> pad to 8 output channels
        co = ow.shape[0]
        self.out_channels = co
        owp = torch.zeros((8, ow.shape[1]), dtype=self.dtype, device=self.device)
        owp[:co] = ow
        obp = torch.zeros((8,), dtype=self.dtype, device=self.device)
        obp[:co] = g("out.2.bias")
        w["out.2.w"], w["out.2.b"] = owp, obp

    def _pack_embeddings(self, g) -> None:
        """time_embed and label_emb; `g(name)` returns the state-dict tensor on the device in the compute dtype."""
        w = self.w
        for p in ("time_embed.0", "time_embed.2"):
            w[p + ".w"], w[p + ".b"] = g(p + ".weight"), g(p + ".bias")
        if self.has_label:
            for p in ("label_emb.0.0", "label_emb.0.2"):
                w[p + ".w"], w[p + ".b"] = g(p + ".weight"), g(p + ".bias")

    def _pack_blocks(self, g, blocks) -> None:
        """Every layer of `blocks` (lists of structure tuples), plus all their ResBlock time-embedding projections stacked
        into one matrix, in block order."""
        w = self.w
        emb_w, emb_b = [], []
        self.emb_off: Dict[str, tuple] = {}
        off = 0

        def pack_layer(layer):
            nonlocal off
            kind, p = layer[0], layer[1]
            if kind == "conv":  # conv_in: Cin=4 -> im2col K=36 padded to 64
                wp = ops.pack_conv3x3(g(p + ".weight"))
                kpad = torch.zeros((wp.shape[0], 64), dtype=self.dtype, device=self.device)
                kpad[:, : wp.shape[1]] = wp
                w[p + ".w"], w[p + ".b"] = kpad, g(p + ".bias")
            elif kind == "res":
                cin, cout = layer[2], layer[3]
                for n in ("in_layers.0", "out_layers.0"):
                    w[f"{p}.{n}.g"], w[f"{p}.{n}.b"] = g(f"{p}.{n}.weight"), g(f"{p}.{n}.bias")
                w[p + ".conv1.w"], w[p + ".conv1.b"] = ops.pack_conv3x3(g(p + ".in_layers.2.weight")), g(p + ".in_layers.2.bias")
                w[p + ".conv2.w"], w[p + ".conv2.b"] = ops.pack_conv3x3(g(p + ".out_layers.3.weight")), g(p + ".out_layers.3.bias")
                emb_w.append(g(p + ".emb_layers.1.weight"))
                emb_b.append(g(p + ".emb_layers.1.bias"))
                self.emb_off[p] = (off, cout)
                off += cout
                if cin != cout:
                    sw = g(p + ".skip_connection.weight")
                    assert sw.shape[2] == 1, "3x3 skip convs (use_conv=True) are not used by SD/SDXL"
                    w[p + ".skip.w"], w[p + ".skip.b"] = sw.reshape(cout, cin).contiguous(), g(p + ".skip_connection.bias")
            elif kind == "attn":
                ch, depth = layer[2], layer[5]
                w[p + ".norm.g"], w[p + ".norm.b"] = g(p + ".norm.weight"), g(p + ".norm.bias")
                for n in ("proj_in", "proj_out"):
                    w[f"{p}.{n}.w"] = g(f"{p}.{n}.weight").reshape(ch, ch).contiguous()
                    w[f"{p}.{n}.b"] = g(f"{p}.{n}.bias")
                heads, dh = layer[3], layer[4]
                # head dims the flash kernels do not take natively (SD1.5: 40 / 80) are zero-padded to 64 / 128 inside
                # the packed projection weights: q.k^T and the kept output columns are unchanged; Dh > 128 (SD1.5: 160)
                # runs through the GEMM-softmax-GEMM path
                dp = dh if dh in (64, 128) else (64 if dh < 64 else (128 if dh < 128 else dh))
                self.head_pad[p] = (dh, dp)

                def pad_rows(wt):  # [H*dh, K] -> [H*dp, K]
                    if dp == dh:
                        return wt
                    o = torch.zeros((heads * dp, wt.shape[1]), dtype=wt.dtype, device=wt.device)
                    o.view(heads, dp, -1)[:, :dh] = wt.view(heads, dh, -1)
                    return o

                def pad_cols(wt):  # [C, H*dh] -> [C, H*dp]
                    if dp == dh:
                        return wt
                    o = torch.zeros((wt.shape[0], heads * dp), dtype=wt.dtype, device=wt.device)
                    o.view(-1, heads, dp)[:, :, :dh] = wt.view(-1, heads, dh)
                    return o

                for d in range(depth):
                    q = f"{p}.transformer_blocks.{d}"
                    # LayerNorm (norm1/2/3, eps 1e-5) is folded into the GEMM that consumes it: weight <- W.gamma,
                    # epilogue y = rstd*(acc - mean*c) + d with the row statistics produced by the previous GEMM
                    gam = {n: g(f"{q}.{n}.weight") for n in ("norm1", "norm2", "norm3")}
                    bet = {n: g(f"{q}.{n}.bias") for n in ("norm1", "norm2", "norm3")}
                    qkv_w = torch.cat([pad_rows(g(f"{q}.attn1.to_q.weight")), pad_rows(g(f"{q}.attn1.to_k.weight")),
                                       pad_rows(g(f"{q}.attn1.to_v.weight"))], 0).contiguous()
                    w[q + ".attn1.qkv"], w[q + ".attn1.qkv.c"], w[q + ".attn1.qkv.d"] = ops.fold_layernorm(qkv_w, None, gam["norm1"], bet["norm1"])
                    w[q + ".attn2.q"], w[q + ".attn2.q.c"], w[q + ".attn2.q.d"] = ops.fold_layernorm(
                        pad_rows(g(f"{q}.attn2.to_q.weight")).contiguous(), None, gam["norm2"], bet["norm2"])
                    w[q + ".attn2.kv"] = torch.cat([pad_rows(g(f"{q}.attn2.to_k.weight")), pad_rows(g(f"{q}.attn2.to_v.weight"))], 0).contiguous()
                    for a in ("attn1", "attn2"):
                        w[f"{q}.{a}.o.w"], w[f"{q}.{a}.o.b"] = pad_cols(g(f"{q}.{a}.to_out.0.weight")).contiguous(), g(f"{q}.{a}.to_out.0.bias")
                    bn = 256 if (4 * ch) % 128 == 0 else 128
                    f1w, f1c, f1d = ops.fold_layernorm(g(f"{q}.ff.net.0.proj.weight"), g(f"{q}.ff.net.0.proj.bias"),
                                                       gam["norm3"], bet["norm3"])
                    w[q + ".ff1.w"], w[q + ".ff1.c"] = ops.pack_geglu(f1w, f1c, bn)   # same row interleave for c and d
                    _, w[q + ".ff1.d"] = ops.pack_geglu(f1w, f1d, bn)
                    w[q + ".ff1.bn"] = bn
                    w[q + ".ff2.w"], w[q + ".ff2.b"] = g(f"{q}.ff.net.2.weight"), g(f"{q}.ff.net.2.bias")
            elif kind == "down":
                w[p + ".w"], w[p + ".b"] = ops.pack_conv3x3(g(p + ".op.weight")), g(p + ".op.bias")
            elif kind == "up":
                # nearest x2 upsample folded into the convolution (four 2x2 parity filters, 16 instead of 36 MACs, no 4x
                # intermediate) whenever the TMA path can slice the channels
                if layer[2] % 64 == 0 and ops.upconv_folded():
                    w[p + ".w4"] = ops.pack_conv3x3_up2x(g(p + ".conv.weight"))
                else:
                    w[p + ".w"] = ops.pack_conv3x3(g(p + ".conv.weight"))
                w[p + ".b"] = g(p + ".conv.bias")

        for blk in blocks:
            for layer in blk:
                pack_layer(layer)
        w["emb_all.w"] = torch.cat(emb_w, 0).contiguous()
        w["emb_all.b"] = torch.cat(emb_b, 0).contiguous()

    # ------------------------------------------------------------------------------------------ blocks
    def _res(self, p: str, layer, x1: torch.Tensor, x2: Optional[torch.Tensor], temb_all: torch.Tensor) -> torch.Tensor:
        w = self.w
        cin, cout = layer[2], layer[3]
        n, hh, ww, c1 = x1.shape
        m = n * hh * ww
        h = ops.groupnorm(x1, w[p + ".in_layers.0.g"], w[p + ".in_layers.0.b"], eps=1e-5, silu=True, x2=x2)
        off, _ = self.emb_off[p]
        h = ops.conv3x3_any(h, w[p + ".conv1.w"], w[p + ".conv1.b"], temb=temb_all[:, off:off + cout])
        h = ops.groupnorm(h, w[p + ".out_layers.0.g"], w[p + ".out_layers.0.b"], eps=1e-5, silu=True)
        if cin != cout:
            skip = ops.gemm(x1.view(m, c1), w[p + ".skip.w"], w[p + ".skip.b"],
                            a2=None if x2 is None else x2.view(m, x2.shape[-1])).view(n, hh, ww, cout)
        else:
            assert x2 is None
            skip = x1
        return ops.conv3x3_any(h, w[p + ".conv2.w"], w[p + ".conv2.b"], residual=skip)

    # ---- cross-attention K/V: the text context is constant over the sampler steps of a job, so its projections
    # (reference: to_k / to_v recomputed in every CrossAttention.forward, unet.py:148-152) are loop-invariant.
    def cross_kv_layers(self):
        out = []
        for blk in self.st["input"] + [self.st["middle"]] + self.st["output"]:
            for layer in blk:
                if layer[0] == "attn":
                    dh, dp = self.head_pad[layer[1]]
                    for d in range(layer[5]):
                        out.append((f"{layer[1]}.transformer_blocks.{d}", layer[3] * dp))
        return out

    def _kv_buffer(self, n: int, n_ctx: int, width: int) -> torch.Tensor:
        # 8 zeroed slack rows: the GEMM-softmax-GEMM path reads the key count rounded up to a multiple of 8
        buf = torch.empty((n * n_ctx + 8, 2 * width), dtype=self.dtype, device=self.device)
        ops.zero_(buf[n * n_ctx:])
        return buf

    def alloc_kv_cache(self, n: int, n_ctx: int) -> Dict[str, torch.Tensor]:
        return {q: self._kv_buffer(n, n_ctx, cw) for q, cw in self.cross_kv_layers()}

    def fill_kv_cache(self, context: torch.Tensor, cache: Dict[str, torch.Tensor]) -> None:
        """One fused K|V projection GEMM per cross-attention layer, once per job."""
        ctx2d = context.view(-1, context.shape[-1])
        for q, _ in self.cross_kv_layers():
            ops.gemm(ctx2d, self.w[q + ".attn2.kv"], out=cache[q][: ctx2d.shape[0]])

    def _attn(self, p: str, layer, x: torch.Tensor, ctx2d: torch.Tensor, n_ctx: int, kv_cache=None) -> torch.Tensor:
        w = self.w
        ch, heads, depth = layer[2], layer[3], layer[5]
        n, hh, ww, _ = x.shape
        L = hh * ww
        m = n * L
        x2d = x.view(m, ch)
        t = ops.groupnorm(x, w[p + ".norm.g"], w[p + ".norm.b"], eps=1e-6, silu=False).view(m, ch)
        # partial row statistics (count, mean, M2) of the residual stream, written by each producer GEMM's epilogue
        st1, st2, st3 = (ops.row_stats_buffer(m, ch, self.device) for _ in range(3))
        t = ops.gemm(t, w[p + ".proj_in.w"], w[p + ".proj_in.b"], row_stats_out=st1)
        dh, dp = self.head_pad[p]
        cw = heads * dp          # width of the (head-padded) q / k / v / attention-output tensors
        scale = dh ** -0.5
        flash = dp in (64, 128)
        nk8 = (n_ctx + 7) // 8 * 8
        for d in range(depth):
            q = f"{p}.transformer_blocks.{d}"
            # self attention
            qkv = ops.gemm(t, w[q + ".attn1.qkv"], ln=(st1, w[q + ".attn1.qkv.c"], w[q + ".attn1.qkv.d"], 1e-5)).view(n, L, 3 * cw)
            if flash:
                att = ops.attention(qkv[:, :, :cw], qkv[:, :, cw:2 * cw], qkv[:, :, 2 * cw:], heads, scale=scale)
            else:
                if (n * L) % 8 == 0:  # one GEMM / block-diagonal softmax / GEMM per head over the whole batch
                    att = ops.attention_blockdiag(qkv[:, :, :cw], qkv[:, :, cw:2 * cw], qkv[:, :, 2 * cw:], heads, scale=scale)
                else:
                    att = ops.attention_generic(qkv[:, :, :cw], qkv[:, :, cw:2 * cw], qkv[:, :, 2 * cw:], heads, scale=scale)
            ops.gemm(att.view(m, cw), w[q + ".attn1.o.w"], w[q + ".attn1.o.b"], residual=t, out=t, row_stats_out=st2)
            # cross attention
            qq = ops.gemm(t, w[q + ".attn2.q"], ln=(st2, w[q + ".attn2.q.c"], w[q + ".attn2.q.d"], 1e-5)).view(n, L, cw)
            if kv_cache is not None:
                kvb = kv_cache[q]
            else:
                kvb = self._kv_buffer(n, n_ctx, cw)
                ops.gemm(ctx2d, w[q + ".attn2.kv"], out=kvb[: n * n_ctx])
            if flash:
                kv = kvb[: n * n_ctx].view(n, n_ctx, 2 * cw)
                att = ops.attention(qq, kv[:, :, :cw], kv[:, :, cw:], heads, scale=scale)
            elif (n * n_ctx) % 8 == 0:
                kv = kvb[: n * n_ctx].view(n, n_ctx, 2 * cw)
                att = ops.attention_blockdiag(qq, kv[:, :, :cw], kv[:, :, cw:], heads, scale=scale)
            else:
                # key count rounded up to 8: the extra rows belong to the next image (or the zeroed slack) and are
                # masked by the softmax (valid_keys), so they contribute exactly 0
                kv = kvb.as_strided((n, nk8, 2 * cw), (n_ctx * 2 * cw, 2 * cw, 1))
                att = ops.attention_generic(qq, kv[:, :, :cw], kv[:, :, cw:], heads, scale=scale, valid_keys=n_ctx)
            ops.gemm(att.view(m, cw), w[q + ".attn2.o.w"], w[q + ".attn2.o.b"], residual=t, out=t, row_stats_out=st3)
            # feed-forward (GEGLU)
            gg = ops.gemm(t, w[q + ".ff1.w"], None, epilogue=EPI_GEGLU, block_n=w[q + ".ff1.bn"],
                          ln=(st3, w[q + ".ff1.c"], w[q + ".ff1.d"], 1e-5))
            ops.gemm(gg, w[q + ".ff2.w"], w[q + ".ff2.b"], residual=t, out=t,
                     row_stats_out=st1 if d + 1 < depth else None)
        out = ops.gemm(t, w[p + ".proj_out.w"], w[p + ".proj_out.b"], residual=x2d)
        return out.view(n, hh, ww, ch)

    def _run(self, layers, h, h2, temb_all, ctx2d, n_ctx, kv_cache=None):
        for layer in layers:
            kind, p = layer[0], layer[1]
            if kind == "res":
                h = self._res(p, layer, h, h2, temb_all)
                h2 = None
            elif kind == "attn":
                h = self._attn(p, layer, h, ctx2d, n_ctx, kv_cache)
            elif kind == "down":
                n, hh, ww, c = h.shape
                cols = ops.im2col3x3(h, stride=2)
                h = ops.gemm(cols, self.w[p + ".w"], self.w[p + ".b"]).view(n, hh // 2, ww // 2, c)
            elif kind == "up":
                if p + ".w4" in self.w:
                    h = ops.conv3x3_up2x(h, self.w[p + ".w4"], self.w[p + ".b"])
                else:
                    h = ops.conv3x3_any(ops.upsample2x(h), self.w[p + ".w"], self.w[p + ".b"])
        return h

    # ------------------------------------------------------------------------------------------ forward
    def _embeddings(self, timesteps: torch.Tensor, y: Optional[torch.Tensor]) -> torch.Tensor:
        w = self.w
        t_emb = ops.timestep_embedding(timesteps, self.mc, self.dtype)
        e = ops.gemm(t_emb, w["time_embed.0.w"], w["time_embed.0.b"], epilogue=EPI_SILU)
        emb = ops.gemm(e, w["time_embed.2.w"], w["time_embed.2.b"])
        if self.has_label:
            assert y is not None
            l1 = ops.gemm(y, w["label_emb.0.0.w"], w["label_emb.0.0.b"], epilogue=EPI_SILU)
            ops.gemm(l1, w["label_emb.0.2.w"], w["label_emb.0.2.b"], residual=emb, out=emb)
        # every ResBlock applies Linear(SiLU(emb)) (unet.py:412-415): one stacked GEMM for all of them
        return ops.gemm(ops.silu(emb), w["emb_all.w"], w["emb_all.b"])

    def control_fits(self, control: dict, n: int, hh: int, ww: int) -> bool:
        """Whether every residual that forward_cols would add for an [n, *, hh, ww] latent is an NCHW tensor of its
        activation's shape, or of batch 1 (added to every image, as the reference's broadcasting `h += ctrl` does), in the
        compute dtype or fp32.  The reference prints "could not be applied" and skips any other residual (apply_control,
        backend/nn/unet.py:44-52): callers hand such calls to Forge's own forward, which does exactly that."""
        shapes = []  # (channels, height, width) after each input block
        c, h, w = self.cfg["in_channels"], hh, ww
        for layers in self.st["input"]:
            for layer in layers:
                if layer[0] in ("conv", "res"):
                    c = layer[3]
                elif layer[0] == "down":
                    h, w = (h + 1) // 2, (w + 1) // 2
            shapes.append((c, h, w))

        def fits(name, wanted):  # wanted: activation shapes in the order the residuals are popped
            lst = list(control.get(name) or [])
            for shp in wanted:
                if not lst:
                    return True
                t = lst.pop()
                if t is not None and not (torch.is_tensor(t) and t.dim() == 4 and t.shape[0] in (n, 1)
                                          and tuple(t.shape[1:]) == shp and t.dtype in (self.dtype, torch.float32)):
                    return False
            return True

        return (fits("input", shapes) and fits("middle", [(c, h, w)])
                and fits("output", shapes[::-1][:len(self.st["output"])]))

    @staticmethod
    def _apply_control(h: torch.Tensor, control: Optional[dict], name: str) -> torch.Tensor:
        """apply_control (backend/nn/unet.py:44-52): pop the LAST tensor of control[name] and add it in place; the
        residual arrives NCHW with h's batch or batch 1 (see control_fits), `h` is channels-last."""
        if control is not None and name in control and len(control[name]) > 0:
            ctrl = control[name].pop()
            if ctrl is not None:
                ops.add_nchw_(h, ctrl.contiguous())
        return h

    def forward_cols(self, cols: torch.Tensor, n: int, hh: int, ww: int, timesteps: torch.Tensor,
                     context: torch.Tensor, y: Optional[torch.Tensor], kv_cache=None, control: Optional[dict] = None) -> torch.Tensor:
        """cols: conv_in im2col rows [n*hh*ww, 64]; returns eps NHWC [n, hh, ww, 8] (channels >= 4 are zero).
        control: ControlNet / T2I-Adapter residuals {"input": [...], "middle": [...], "output": [...]} of NCHW tensors, consumed
        from the end of each list exactly as the reference does (unet.py:714, 733, 739)."""
        w = self.w
        assert context.dtype == self.dtype and context.is_contiguous() and context.shape[0] == n
        n_ctx = context.shape[1]
        ctx2d = context.view(n * n_ctx, context.shape[2])
        temb_all = self._embeddings(timesteps, y)
        if control is not None:
            control = {k: list(v) for k, v in control.items()}  # the lists are consumed; leave the caller's intact
        p0 = self.st["input"][0][0][1]
        h = ops.gemm(cols, w[p0 + ".w"], w[p0 + ".b"]).view(n, hh, ww, self.mc)
        h = self._apply_control(h, control, "input")
        hs = [h]
        for layers in self.st["input"][1:]:
            h = self._run(layers, h, None, temb_all, ctx2d, n_ctx, kv_cache)
            h = self._apply_control(h, control, "input")
            hs.append(h)
        h = self._run(self.st["middle"], h, None, temb_all, ctx2d, n_ctx, kv_cache)
        h = self._apply_control(h, control, "middle")
        for layers in self.st["output"]:
            h = self._run(layers, h, self._apply_control(hs.pop(), control, "output"), temb_all, ctx2d, n_ctx, kv_cache)
        h = ops.groupnorm(h, w["out.0.g"], w["out.0.b"], eps=1e-5, silu=True)
        return ops.conv3x3_any(h, w["out.2.w"], w["out.2.b"])

    def forward(self, x: torch.Tensor, timesteps: torch.Tensor, context: torch.Tensor,
                y: Optional[torch.Tensor] = None, control: Optional[dict] = None) -> torch.Tensor:
        """Same contract as IntegratedUNet2DConditionModel.forward (unet.py:696): x NCHW [N,4,h,w] in the
        computation dtype, timesteps [N], context [N,77,ctx], y [N,adm] -> NCHW [N,4,h,w]."""
        n, c, hh, ww = x.shape
        xn = ops.nchw_to_nhwc(x.to(self.dtype).contiguous(), self.dtype)
        cols = ops.im2col3x3(xn, ldo=64)
        eps = self.forward_cols(cols, n, hh, ww, timesteps.float().contiguous(), context.to(self.dtype).contiguous(),
                                None if y is None else y.to(self.dtype).contiguous(), control=control)
        return ops.nhwc_to_nchw(eps, channels=self.out_channels, out_dtype=x.dtype)

    def supports_latent(self, hh: int, ww: int) -> bool:
        """True when every resolution level of the UNet tiles on the TMA convolution path (ops.conv3x3_supported) and the
        stride-2 downsamples are exact.  1024x1024 / 512x512 and the other power-of-two sizes do; SDXL's non-square
        buckets (e.g. 152x104 latents) do not yet — the plug-in hands those back to Forge's own forward."""
        levels = len(self.cfg["channel_mult"])
        for _ in range(levels):
            if not (ops.conv3x3_supported(hh, ww) or ops.any_size_enabled()):
                return False
            if _ != levels - 1:
                if hh % 2 or ww % 2:
                    return False
                hh, ww = hh // 2, ww // 2
        return True

    def forward_sigma(self, x: torch.Tensor, sigma: torch.Tensor, timesteps: torch.Tensor, context: torch.Tensor,
                      y: Optional[torch.Tensor], reps: int, kv_cache=None, control: Optional[dict] = None) -> torch.Tensor:
        """KModel.apply_model's front half fused into the entry (k_model.py:27-36): x fp32 NCHW [B,4,h,w] is
        scaled by 1/sqrt(sigma^2+1), cast, laid out channels-last and replicated `reps` times (cond/uncond
        batch) in one pass.  Returns eps NHWC [reps*B, h, w, 8]."""
        b, c, hh, ww = x.shape
        cols = ops.unet_input_im2col(x, sigma, self.dtype, reps=reps, ldo=64)
        return self.forward_cols(cols, reps * b, hh, ww, timesteps, context, y, kv_cache, control)
