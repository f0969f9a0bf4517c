"""Tensor-level wrappers over the C ABI: torch tensors in, raw pointers + descriptors out.

PyTorch is used for device memory and streams only; every function here enqueues exactly the
hand-written sm_100a kernels of libb200forge.so on the current CUDA stream.  Nothing in this module
falls back to a torch op — unsupported shapes raise `B200Error` (code B200_EUNSUPPORTED) so that the
caller (the plug-in layer) can decide to hand the block back to Forge's own code.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import lib as _l
from .lib import (B200Error, EPI_GEGLU, EPI_GELU, EPI_GELU_TANH, EPI_NONE, EPI_SILU, STEP_DPMPP_2M, STEP_EULER, STEP_LINEAR)  # noqa: F401

LAUNCHES = 0  # kernels enqueued through this module (bench.py reports it as gpu_launches)
PROFILE = None  # set to a list to record (family, algorithmic flops, algorithmic bytes, start_evt, end_evt) per call


class _prof:
    """CUDA-event bracket around one library call on the launching stream (bench.py roofline accounting)."""

    def __init__(self, family: str, flops: float = 0.0, nbytes: float = 0.0, label: str = ""):
        self.family, self.flops, self.nbytes, self.label = family, flops, nbytes, label

    def __enter__(self):
        if PROFILE is not None:
            self.s = torch.cuda.Event(enable_timing=True)
            self.s.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            PROFILE.append((self.family, self.flops, self.nbytes, self.s, e, self.label))
        return False


def _count(n: int = 1) -> None:
    global LAUNCHES
    LAUNCHES += n


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float16:
        return _l.B200_F16
    if t.dtype == torch.bfloat16:
        return _l.B200_BF16
    raise TypeError(f"b200forge kernels take fp16/bf16 tensors, got {t.dtype}")


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _rowmajor2d(t: torch.Tensor, name: str) -> None:
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError(f"{name}: expected a 2-D tensor with unit inner stride, got {tuple(t.shape)} / {t.stride()}")


_WS: dict = {}


def gemm_workspace(device: torch.device) -> int:
    """Scratch buffer of the GEMM / convolution K-split (b200_gemm_desc.workspace) for the CURRENT stream of `device`: one
    zero-initialised buffer per (device, stream) — launches on one stream never overlap, launches on different streams get
    different buffers.  Allocated through torch's caching allocator, so a first use inside a CUDA-graph capture is legal (the
    block then lives in the graph's pool for as long as this cache holds it)."""
    st = torch.cuda.current_stream(device)
    key = (st.device.index, st.cuda_stream)
    t = _WS.get(key)
    if t is None:
        t = torch.zeros(_l.load().b200_gemm_workspace_bytes(), dtype=torch.uint8, device=st.device)
        _WS[key] = t
    return t.data_ptr()


def gemm(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, *,
         residual: Optional[torch.Tensor] = None, rowvec: Optional[torch.Tensor] = None, rows_per_vec: int = 1,
         epilogue: int = EPI_NONE, a2: Optional[torch.Tensor] = None, bias_along_m: bool = False,
         out: Optional[torch.Tensor] = None, block_n: int = 0, ln: Optional[tuple] = None,
         row_stats_out: Optional[torch.Tensor] = None, rowvec_mul: bool = False, act_col0: int = 0,
         seg: Optional[tuple] = None, alpha: float = 1.0) -> torch.Tensor:
    """out[M, N] = epi(alpha * cat(a, a2) @ w.T + bias + rowvec[row // rows_per_vec]) + residual.

    a [M, K1], a2 [M, K2] (optional), w [N, K1+K2] — all with unit inner stride (row strides free).
    GEGLU: w/bias rows must be pre-interleaved with `pack_geglu`; out is [M, N/2].
    ln = (stats [P,M,4] fp32, c [N] fp32, d [N] fp32, eps): LayerNorm of `a` folded into the GEMM (w must be W*gamma,
    see `fold_layernorm`); stats = the partial row statistics a producer GEMM wrote.  row_stats_out [P,M,4] fp32
    (`row_stats_buffer`; nothing to zero): receives partial (count, mean, M2) statistics of the output rows.
    rowvec_mul: out = residual + rowvec * (acc + bias) (modulation gate).  act_col0: the activation applies to output
    columns >= act_col0.  seg = (period, split, w2, bias2, rowvec2): rows with (m % period) >= split use the second
    weight set (Flux double-stream blocks on the joint [txt | img] activation).
    """
    _rowmajor2d(a, "a")
    _rowmajor2d(w, "w")
    M, K1 = a.shape
    N, K = w.shape
    if a2 is not None:
        _rowmajor2d(a2, "a2")
        assert a2.shape[0] == M and K1 + a2.shape[1] == K
    else:
        assert K1 == K, (a.shape, w.shape)
    n_out = N // 2 if epilogue == EPI_GEGLU else N
    if out is None:
        out = torch.empty((M, n_out), dtype=a.dtype, device=a.device)
    _rowmajor2d(out, "out")
    assert out.shape[0] == M and out.shape[1] == n_out
    d = _l.GemmDesc()
    d.M, d.N, d.K = M, N, K
    d.workspace = gemm_workspace(a.device)
    d.lda, d.ldb, d.ldc = a.stride(0), w.stride(0), out.stride(0)
    d.dtype = _dt(a)
    d.epilogue = epilogue
    d.block_n = block_n
    d.bias = _p(bias)
    d.bias_along_m = 1 if bias_along_m else 0
    if residual is not None:
        _rowmajor2d(residual, "residual")
        d.residual, d.ldr = residual.data_ptr(), residual.stride(0)
    if rowvec is not None:
        _rowmajor2d(rowvec, "rowvec")
        d.rowvec, d.ld_rowvec, d.rows_per_vec = rowvec.data_ptr(), rowvec.stride(0), rows_per_vec
    if a2 is not None:
        d.A2, d.lda2, d.K1 = a2.data_ptr(), a2.stride(0), K1
    if ln is not None:
        st, lc, ld_, eps = ln
        assert st.dtype == torch.float32 and st.dim() == 3 and st.shape[1] == M and st.shape[2] == 4 and st.is_contiguous()
        assert lc.dtype == torch.float32 and ld_.dtype == torch.float32 and lc.numel() == N and ld_.numel() == N
        d.ln_stats, d.ln_stats_parts, d.ln_c, d.ln_d, d.ln_eps = st.data_ptr(), st.shape[0], lc.data_ptr(), ld_.data_ptr(), eps
    if row_stats_out is not None:
        assert row_stats_out.dtype == torch.float32 and row_stats_out.is_contiguous()
        assert tuple(row_stats_out.shape) == (row_stats_parts(N, epilogue, block_n), M, 4), (row_stats_out.shape, N)
        d.row_stats_out = row_stats_out.data_ptr()
    d.rowvec_mul = 1 if rowvec_mul else 0
    d.act_col0 = act_col0
    d.alpha = float(alpha)
    if seg is not None:
        period, split, w2, bias2, rowvec2 = seg
        _rowmajor2d(w2, "w2")
        assert w2.shape == w.shape and w2.stride(0) == w.stride(0)
        assert rowvec2 is None or rowvec2.stride(0) == rowvec.stride(0)
        d.B2, d.bias2, d.rowvec2 = w2.data_ptr(), _p(bias2), _p(rowvec2)
        d.seg_period, d.seg_split = period, split
    with _prof("gemm", 2.0 * M * N * K, 2.0 * (M * K + N * K + M * n_out),
               f"gemm M={M} N={N} K={K}" + (" ln" if ln is not None else "") + (" stats" if row_stats_out is not None else "") +
               (" geglu" if epilogue == EPI_GEGLU else "") + (" res" if residual is not None else "") + (" a2" if a2 is not None else "")
               if PROFILE is not None else ""):
        _l.check(_l.load().b200_gemm(a.data_ptr(), w.data_ptr(), out.data_ptr(), C.byref(d), _stream()))
    _count()
    return out


def row_stats_parts(N: int, epilogue: int = EPI_NONE, block_n: int = 0) -> int:
    """Partials per row that a GEMM with N output columns writes to `row_stats_out` (2 per N tile)."""
    return int(_l.load().b200_gemm_row_stats_parts(N, epilogue, block_n))


def row_stats_buffer(M: int, N: int, device, epilogue: int = EPI_NONE, block_n: int = 0) -> torch.Tensor:
    """[P, M, 4] fp32 buffer for `gemm(..., row_stats_out=)` (part-major: a warp's 32 rows of one part are contiguous); every
    partial is overwritten by the GEMM (no zero-fill)."""
    return torch.empty((row_stats_parts(N, epilogue, block_n), M, 4), dtype=torch.float32, device=device)


def pack_geglu(w: torch.Tensor, b: Optional[torch.Tensor], block_n: int = 256):
    """Interleave GEGLU projection rows so each BN-wide output tile holds BN/2 value rows followed by
    the matching BN/2 gate rows (reference layout: rows [0, I) value, [I, 2I) gate — unet.py:109-110)."""
    two_i = w.shape[0]
    inner = two_i // 2
    half = block_n // 2
    assert inner % half == 0, (inner, block_n)
    idx = torch.arange(two_i, device=w.device).view(-1, block_n)
    tile = idx // block_n
    within = idx % block_n
    src = torch.where(within < half, tile * half + within, inner + tile * half + (within - half)).reshape(-1)
    wp = w.index_select(0, src).contiguous()
    bp = b.index_select(0, src).contiguous() if b is not None else None
    return wp, bp


def fold_layernorm(w: torch.Tensor, b: Optional[torch.Tensor], gamma: torch.Tensor, beta: torch.Tensor):
    """LayerNorm -> Linear as one GEMM on the raw rows:  LN(x) W^T + b = rstd (x (W.gamma)^T - mean c) + d,
    c = rowsum(W.gamma), d = W beta + b.  Returns (W.gamma in the weight dtype, c fp32, d fp32); c is summed from the
    *rounded* folded weight so that it cancels exactly against what the tensor core multiplies."""
    wf = (w.float() * gamma.float()[None, :]).to(w.dtype).contiguous()
    c = wf.float().sum(dim=1).contiguous()
    d = (w.float() @ beta.float())
    if b is not None:
        d = d + b.float()
    return wf, c, d.contiguous()


def refresh_packed(old: dict, new: dict) -> dict:
    """Engine re-pack after the source module's weights changed (LoRA merge): copy the freshly packed tensors INTO the old
    buffers wherever shape and dtype agree, so device addresses — which captured CUDA graphs hold — stay valid."""
    out = {}
    for k, v in new.items():
        o = old.get(k)
        if torch.is_tensor(v) and torch.is_tensor(o) and o.shape == v.shape and o.dtype == v.dtype and o.device == v.device:
            o.copy_(v)
            out[k] = o
        else:
            out[k] = v
    return out


def zero_(t: torch.Tensor) -> torch.Tensor:
    assert t.is_contiguous()
    _l.check(_l.load().b200_fill_zero(t.data_ptr(), t.numel() * t.element_size(), _stream()))
    return t


def pack_conv3x3(w: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, 3, 3] (torch Conv2d) -> [Cout, 9*Cin] with k = (ky*3 + kx)*Cin + c."""
    co, ci, kh, kw = w.shape
    assert kh == 3 and kw == 3
    return w.permute(0, 2, 3, 1).reshape(co, 9 * ci).contiguous()


def conv3x3_supported(h: int, w: int) -> bool:
    """Whether b200_conv3x3 can tile an [*, h, w, *] image: 128 output pixels per tile must form a box of whole rows
    (w a power of two <= 128 with h a multiple of 128 // w, or the whole image when it has fewer than 128 pixels) or a
    128-pixel row segment (w a multiple of 128).  Mirrors the host checks in csrc/gemm.cu."""
    tile_w = w if w < 128 else 128
    if 128 % tile_w or w % tile_w:
        return False
    tile_h = min(128 // tile_w, h)
    if h % tile_h or 128 % (tile_w * tile_h):
        return False
    tile_n = 128 // (tile_w * tile_h)
    return tile_n == 1 or (tile_w == w and tile_h == h)


def conv3x3(x1: torch.Tensor, w_packed: torch.Tensor, bias: Optional[torch.Tensor] = None, *,
            x2: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
            temb: Optional[torch.Tensor] = None, epilogue: int = EPI_NONE, out: Optional[torch.Tensor] = None,
            block_n: int = 0) -> torch.Tensor:
    """3x3/stride 1/pad 1 convolution on contiguous NHWC tensors; x2 is an optional second channel group."""
    assert x1.dim() == 4 and x1.is_contiguous()
    n, h, w_, c1 = x1.shape
    c2 = 0
    if x2 is not None:
        assert x2.is_contiguous() and x2.shape[:3] == x1.shape[:3]
        c2 = x2.shape[3]
    cout = w_packed.shape[0]
    assert w_packed.shape[1] == 9 * (c1 + c2) and w_packed.is_contiguous()
    if out is None:
        out = torch.empty((n, h, w_, cout), dtype=x1.dtype, device=x1.device)
    assert out.is_contiguous()
    d = _l.Conv3x3Desc()
    d.N, d.H, d.W, d.C1, d.C2, d.Cout = n, h, w_, c1, c2, cout
    d.workspace = gemm_workspace(x1.device)
    d.dtype = _dt(x1)
    d.epilogue = epilogue
    d.block_n = block_n
    d.bias = _p(bias)
    if residual is not None:
        assert residual.is_contiguous()
        d.residual, d.ldr = residual.data_ptr(), residual.shape[-1]
    if temb is not None:
        _rowmajor2d(temb, "temb")
        d.temb, d.ld_temb = temb.data_ptr(), temb.stride(0)
    with _prof("conv3x3", 2.0 * n * h * w_ * cout * 9 * (c1 + c2), 2.0 * (n * h * w_ * (c1 + c2 + cout) + cout * 9 * (c1 + c2)),
               f"conv {n}x{h}x{w_} {c1}+{c2}->{cout}" + (" res" if residual is not None else "") + (" temb" if temb is not None else "")):
        _l.check(_l.load().b200_conv3x3(x1.data_ptr(), _p(x2), w_packed.data_ptr(), out.data_ptr(), C.byref(d), _stream()))
    _count()
    return out


def pack_conv3x3_up2x(w: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> [4*Cout, 4*Cin] for b200_conv3x3_up2x: the 3x3 filter applied to a nearest-x2-upsampled image
    is, for output parity (py, px), a 2x2 filter on the low-res image whose taps are sums of the original ones
    (rows {0 | 1+2} for py = 0, {0+1 | 2} for py = 1; same for columns).  Row (py*2+px)*Cout + co, k = (ty*2+tx)*Cin + c;
    sums in fp32, rounded once to the weight dtype."""
    co, ci, kh, kw = w.shape
    assert kh == 3 and kw == 3
    wf = w.float()
    sets = (((0,), (1, 2)), ((0, 1), (2,)))  # sets[parity][tap] = original taps folded into it
    out = torch.empty((2, 2, co, 2, 2, ci), dtype=torch.float32, device=w.device)
    for py in range(2):
        for px in range(2):
            for ty in range(2):
                for tx in range(2):
                    acc = torch.zeros((co, ci), dtype=torch.float32, device=w.device)
                    for ky in sets[py][ty]:
                        for kx in sets[px][tx]:
                            acc = acc + wf[:, :, ky, kx]
                    out[py, px, :, ty, tx, :] = acc
    return out.reshape(4 * co, 4 * ci).to(w.dtype).contiguous()


def upconv_folded() -> bool:
    """B200_UPCONV=0: upsample2x + conv3x3 (4x tensor materialised, 36 MACs) instead of the folded b200_conv3x3_up2x."""
    import os
    return os.environ.get("B200_UPCONV", "1") != "0"


def conv3x3_up2x(x: torch.Tensor, w_packed4: torch.Tensor, bias: Optional[torch.Tensor] = None, *,
                 epilogue: int = EPI_NONE, out: Optional[torch.Tensor] = None, block_n: int = 0) -> torch.Tensor:
    """conv3x3(upsample2x(x)) on a contiguous NHWC tensor without the 4x intermediate (w_packed4 from pack_conv3x3_up2x);
    x [N, H, W, C] with C a multiple of 64, any H, W -> [N, 2H, 2W, Cout]."""
    assert x.dim() == 4 and x.is_contiguous()
    n, h, w_, c = x.shape
    cout = w_packed4.shape[0] // 4
    assert w_packed4.shape == (4 * cout, 4 * c) and w_packed4.is_contiguous() and c % 64 == 0
    if out is None:
        out = torch.empty((n, 2 * h, 2 * w_, cout), dtype=x.dtype, device=x.device)
    assert out.is_contiguous() and out.shape == (n, 2 * h, 2 * w_, cout)
    d = _l.Conv3x3Desc()
    d.N, d.H, d.W, d.C1, d.C2, d.Cout = n, h, w_, c, 0, cout
    d.workspace = gemm_workspace(x.device)
    d.dtype = _dt(x)
    d.epilogue = epilogue
    d.block_n = block_n
    d.bias = _p(bias)
    # FLOPs actually executed (16 MACs per output pixel and channel pair); the reference's upsample + conv does 36
    with _prof("conv3x3", 2.0 * n * 4 * h * w_ * cout * 4 * c, 2.0 * (n * h * w_ * (c + 4 * cout) + cout * 16 * c),
               f"conv-up2x {n}x{h}x{w_} {c}->{cout}"):
        _l.check(_l.load().b200_conv3x3_up2x(x.data_ptr(), None, w_packed4.data_ptr(), out.data_ptr(), C.byref(d), _stream()))
    _count()
    return out


def conv_route() -> str:
    """How 3x3 convolutions of images that do not tile into 128-pixel TMA boxes run (B200_CONV_ROUTE):
      generic (default)  inside the implicit-GEMM kernel with overhanging tiles and masked stores (FEAT = 4 build);
      im2col             patch matrix (b200_im2col3x3) + b200_gemm with the same epilogue — 9x the activation traffic;
      exact              not at all: such sizes raise B200_EUNSUPPORTED / are handed back to Forge (the round-1 behaviour)."""
    import os
    r = os.environ.get("B200_CONV_ROUTE", "generic")
    if r not in ("generic", "im2col", "exact"):
        raise ValueError(f"B200_CONV_ROUTE={r!r}: generic | im2col | exact")
    return r


def any_size_enabled() -> bool:
    """Whether image sizes outside `conv3x3_supported` are served by the fused engines (see `conv_route`)."""
    return conv_route() != "exact"


def conv3x3_any(x: torch.Tensor, w_packed: torch.Tensor, bias: Optional[torch.Tensor] = None, *,
                residual: Optional[torch.Tensor] = None, temb: Optional[torch.Tensor] = None, epilogue: int = EPI_NONE,
                out: Optional[torch.Tensor] = None, route: Optional[str] = None) -> torch.Tensor:
    """3x3 / stride 1 / pad 1 on one contiguous NHWC tensor for ANY image size: the implicit-GEMM TMA kernel when the size
    tiles exactly (conv3x3_supported) or through its generic tiling, else patch matrix + GEMM with the same epilogue (bias,
    per-image time-embedding row, activation, residual)."""
    n, h, w_, c = x.shape
    route = route or conv_route()
    if c % 64 == 0 and (conv3x3_supported(h, w_) or route == "generic"):  # the TMA path slices channels in 64s
        return conv3x3(x, w_packed, bias, residual=residual, temb=temb, epilogue=epilogue, out=out)
    if route == "exact" and c % 64 == 0:
        raise B200Error(_l.E_UNSUPPORTED, f"conv3x3: {h}x{w_} does not tile into 128-pixel boxes (B200_CONV_ROUTE=exact)")
    cout = w_packed.shape[0]
    if out is None:
        out = torch.empty((n, h, w_, cout), dtype=x.dtype, device=x.device)
    cols = im2col3x3(x)
    gemm(cols, w_packed, bias, rowvec=temb, rows_per_vec=h * w_, epilogue=epilogue,
         residual=None if residual is None else residual.reshape(n * h * w_, cout), out=out.view(n * h * w_, cout))
    return out


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, *, scale: Optional[float] = None,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q [B, Lq, H*Dh], k/v [B, Lk, H*Dh] (unit inner stride; may be column slices of a fused projection)."""
    b, lq, hd = q.shape
    lk = k.shape[1]
    dh = hd // heads
    for t in (q, k, v):
        assert t.dim() == 3 and t.stride(2) == 1 and t.shape[2] == hd
    if out is None:
        out = torch.empty((b, lq, hd), dtype=q.dtype, device=q.device)
    assert out.stride(2) == 1
    d = _l.AttnDesc()
    d.B, d.H, d.Lq, d.Lk, d.Dh = b, heads, lq, lk, dh
    d.q_stride_b, d.q_stride_l = q.stride(0), q.stride(1)
    d.k_stride_b, d.k_stride_l = k.stride(0), k.stride(1)
    d.v_stride_b, d.v_stride_l = v.stride(0), v.stride(1)
    d.o_stride_b, d.o_stride_l = out.stride(0), out.stride(1)
    d.scale = float(scale if scale is not None else dh ** -0.5)
    d.dtype = _dt(q)
    with _prof("attention", 4.0 * b * heads * lq * lk * dh, 2.0 * b * hd * (2 * lq + 2 * lk), f"attn B={b} H={heads} Lq={lq} Lk={lk} Dh={dh}"):
        _l.check(_l.load().b200_attention(q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), C.byref(d), _stream()))
    _count()
    return out


def attention_generic(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, *, scale: float,
                      valid_keys: Optional[int] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Any head dim (multiple of 8), any key count padded to a multiple of 8 (`valid_keys` real ones): per (batch, head)
    S = Q K^T (GEMM) -> masked row softmax -> O = P V (GEMM against V^T).  Used for SD1.5's Dh = 160 levels
    (64 / 256 tokens), where a dedicated flash kernel is not worth its shared-memory footprint."""
    b, lq, hd = q.shape
    lk = k.shape[1]
    dh = hd // heads
    assert dh % 8 == 0 and lk % 8 == 0 and all(t.stride(2) == 1 for t in (q, k, v))
    if out is None:
        out = torch.empty((b, lq, hd), dtype=q.dtype, device=q.device)
    s = torch.empty((lq, lk), dtype=q.dtype, device=q.device)
    for i in range(b):
        vt = transpose_rows(v[i])  # V^T [H*dh, Lk]
        for h in range(heads):
            sl = slice(h * dh, (h + 1) * dh)
            gemm(q[i, :, sl], k[i, :, sl], out=s, alpha=scale)  # scaled logits: the unscaled ones can leave the fp16 range
            softmax_rows_(s, 1.0, valid_keys)
            gemm(s, vt[sl], out=out[i, :, sl])
    return out


def attention_blockdiag(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, heads: int, *, scale: float,
                        out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Any head dim (multiple of 8) and any key count, batched over the samples: per head ONE S = Q_h K_h^T over the
    whole batch [B*Lq, B*Lk], a block-diagonal row softmax (each sample's rows keep only their own keys) and ONE
    O_h = P V_h — 3 launches per head instead of 3 per (sample, head).  q [B, Lq, H*Dh]; k, v [B, Lk, H*Dh] whose batch
    stride equals Lk rows (so [B*Lk, H*Dh] is one matrix); B*Lk must be a multiple of 8."""
    b, lq, hd = q.shape
    lk = k.shape[1]
    dh = hd // heads
    assert dh % 8 == 0 and (b * lk) % 8 == 0
    for t, L in ((q, lq), (k, lk), (v, lk)):
        assert t.stride(2) == 1 and t.stride(0) == L * t.stride(1), "batch must be contiguous in rows"
    q2 = q.as_strided((b * lq, hd), (q.stride(1), 1))
    k2 = k.as_strided((b * lk, hd), (k.stride(1), 1))
    v2 = v.as_strided((b * lk, hd), (v.stride(1), 1))
    if out is None:
        out = torch.empty((b, lq, hd), dtype=q.dtype, device=q.device)
    o2 = out.view(b * lq, hd)
    vt = transpose_rows(v2)  # V^T [H*Dh, B*Lk]
    s = torch.empty((b * lq, b * lk), dtype=q.dtype, device=q.device)
    for h in range(heads):
        sl = slice(h * dh, (h + 1) * dh)
        gemm(q2[:, sl], k2[:, sl], out=s, alpha=scale)  # scaled logits (see attention_generic)
        _l.check(_l.load().b200_softmax_rows_blockdiag(s.data_ptr(), b * lq, b * lk, s.stride(0), 1.0, lq, lk, lk,
                                                       _dt(s), _stream()))
        _count()
        gemm(s, vt[sl], out=o2[:, sl])
    return out


_GN_WS: dict = {}  # device index -> zero-initialised workspace shared by all stream-ordered GroupNorm calls
_GN_WS_BYTES = 4 << 20


def gn_workspace(device) -> torch.Tensor:
    """The GroupNorm workspace of `device` (ticket counters + statistics, b200_groupnorm_ws_bytes).  Created zeroed on
    first use — engines call this at construction so that it never happens inside a CUDA-graph capture; the kernel resets
    its counters, so the buffer is never zeroed again."""
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    ws = _GN_WS.get(idx)
    if ws is None:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("groupnorm workspace must be created before CUDA-graph capture (ops.gn_workspace(device))")
        ws = torch.zeros((_GN_WS_BYTES,), dtype=torch.uint8, device=torch.device("cuda", idx))
        _GN_WS[idx] = ws
    return ws


def groupnorm(x1: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, *, groups: int = 32, eps: float = 1e-5,
              silu: bool = False, x2: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GroupNorm(+SiLU) over the channel concat of NHWC tensors x1, x2 -> NHWC [.., C1+C2].  Two launches (deterministic
    statistics, apply); bit-reproducible run to run."""
    assert x1.is_contiguous()
    n = x1.shape[0]
    c1 = x1.shape[-1]
    hw = x1.numel() // (n * c1)
    c2 = 0
    if x2 is not None:
        assert x2.is_contiguous() and x2.shape[:-1] == x1.shape[:-1]
        c2 = x2.shape[-1]
    if out is None:
        out = torch.empty(tuple(x1.shape[:-1]) + (c1 + c2,), dtype=x1.dtype, device=x1.device)
    d = _l.GnDesc()
    d.N, d.HW, d.C1, d.C2, d.groups, d.eps, d.silu, d.dtype = n, hw, c1, c2, groups, eps, 1 if silu else 0, _dt(x1)
    L = _l.load()
    st = _stream()
    ws = gn_workspace(x1.device)
    if L.b200_groupnorm_ws_bytes(C.byref(d)) > ws.numel():
        raise B200Error(_l.E_UNSUPPORTED, f"groupnorm: batch {n} x {groups} groups exceeds the {ws.numel()}-byte workspace")
    with _prof("groupnorm", 0.0, 2.0 * 3 * n * hw * (c1 + c2), f"gn {n}x{hw}x{c1}+{c2}"):
        _l.check(L.b200_groupnorm_stats(x1.data_ptr(), _p(x2), ws.data_ptr(), C.byref(d), st))
        _l.check(L.b200_groupnorm_apply(x1.data_ptr(), _p(x2), ws.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                        out.data_ptr(), C.byref(d), st))
    _count(2)
    return out


def layernorm(x: torch.Tensor, gamma: Optional[torch.Tensor], beta: Optional[torch.Tensor], eps: float = 1e-5,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    assert x.is_contiguous()
    c = x.shape[-1]
    rows = x.numel() // c
    if out is None:
        out = torch.empty_like(x)
    with _prof("layernorm", 0.0, 2.0 * 2 * rows * c):
        _l.check(_l.load().b200_layernorm(x.data_ptr(), _p(gamma), _p(beta), out.data_ptr(), rows, c, eps, _dt(x), _stream()))
    _count()
    return out


def upsample2x(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    assert x.dim() == 4 and x.is_contiguous()
    n, h, w, c = x.shape
    if out is None:
        out = torch.empty((n, 2 * h, 2 * w, c), dtype=x.dtype, device=x.device)
    _l.check(_l.load().b200_upsample2x(x.data_ptr(), out.data_ptr(), n, h, w, c, _dt(x), _stream()))
    _count()
    return out


def im2col3x3(x: torch.Tensor, *, stride: int = 1, pad_lo: int = 1, pad_hi: int = 1, ldo: Optional[int] = None,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """NHWC -> [N*Ho*Wo, ldo] patch matrix, k = (ky*3+kx)*C + c, zero padded to ldo columns."""
    assert x.dim() == 4 and x.is_contiguous()
    n, h, w, c = x.shape
    ho = (h + pad_lo + pad_hi - 3) // stride + 1
    wo = (w + pad_lo + pad_hi - 3) // stride + 1
    if ldo is None:
        ldo = (9 * c + 7) // 8 * 8
    if out is None:
        out = torch.empty((n * ho * wo, ldo), dtype=x.dtype, device=x.device)
    _l.check(_l.load().b200_im2col3x3(x.data_ptr(), out.data_ptr(), n, h, w, c, stride, pad_lo, ho, wo, ldo, _dt(x),
                                      _stream()))
    _count()
    return out


def nchw_to_nhwc(x: torch.Tensor, dtype: torch.dtype, *, ldy: Optional[int] = None, scale: float = 1.0,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """NCHW (fp32 or `dtype`) -> NHWC `dtype` with optional scaling and zero channel padding to ldy."""
    assert x.dim() == 4 and x.is_contiguous()
    n, c, h, w = x.shape
    ldy = ldy or c
    if out is None:
        out = torch.empty((n, h, w, ldy), dtype=dtype, device=x.device)
    is_f32 = x.dtype == torch.float32
    assert is_f32 or x.dtype == dtype
    _l.check(_l.load().b200_nchw_to_nhwc(x.data_ptr(), out.data_ptr(), n, c, h, w, ldy, scale, 1 if is_f32 else 0,
                                         _dt(out), _stream()))
    _count()
    return out


def nhwc_to_nchw(x: torch.Tensor, channels: Optional[int] = None, out_dtype: Optional[torch.dtype] = None,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x NHWC (channel stride ldx = x.shape[3]); keeps the first `channels` channels."""
    assert x.dim() == 4 and x.is_contiguous()
    n, h, w, ldx = x.shape
    c = channels or ldx
    out_dtype = out_dtype or x.dtype
    if out is None:
        out = torch.empty((n, c, h, w), dtype=out_dtype, device=x.device)
    _l.check(_l.load().b200_nhwc_to_nchw(x.data_ptr(), out.data_ptr(), n, c, h, w, ldx,
                                         1 if out.dtype == torch.float32 else 0, _dt(x), _stream()))
    _count()
    return out


def transpose_rows(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[L, C] (unit inner stride, any row stride) -> contiguous [C, L]; the NHWC->NCHW kernel with H = L, W = 1."""
    _rowmajor2d(x, "x")
    L, c = x.shape
    if out is None:
        out = torch.empty((c, L), dtype=x.dtype, device=x.device)
    _l.check(_l.load().b200_nhwc_to_nchw(x.data_ptr(), out.data_ptr(), 1, c, L, 1, x.stride(0), 0, _dt(x), _stream()))
    _count()
    return out


def silu(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    assert x.is_contiguous()
    if out is None:
        out = torch.empty_like(x)
    _l.check(_l.load().b200_silu(x.data_ptr(), out.data_ptr(), x.numel(), _dt(x), _stream()))
    _count()
    return out


def softmax_rows_(x: torch.Tensor, scale: float, valid_cols: Optional[int] = None) -> torch.Tensor:
    _rowmajor2d(x, "x")
    _l.check(_l.load().b200_softmax_rows(x.data_ptr(), x.shape[0], x.shape[1], valid_cols or x.shape[1], x.stride(0),
                                         scale, _dt(x), _stream()))
    _count()
    return x


def timestep_embedding(t: torch.Tensor, dim: int, dtype: torch.dtype, max_period: float = 10000.0,
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
    assert t.dtype == torch.float32 and t.is_contiguous()
    if out is None:
        out = torch.empty((t.shape[0], dim), dtype=dtype, device=t.device)
    _l.check(_l.load().b200_timestep_embedding(t.data_ptr(), out.data_ptr(), t.shape[0], dim, max_period, _dt(out), _stream()))
    _count()
    return out


def unet_input_im2col(x: torch.Tensor, sigma: torch.Tensor, dtype: torch.dtype, *, reps: int, ldo: int,
                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
    assert x.dtype == torch.float32 and x.is_contiguous() and sigma.dtype == torch.float32
    b, c, h, w = x.shape
    if out is None:
        out = torch.empty((reps * b * h * w, ldo), dtype=dtype, device=x.device)
    _l.check(_l.load().b200_unet_input_im2col(x.data_ptr(), sigma.data_ptr(), out.data_ptr(), b, c, h, w, ldo, reps,
                                              _dt(out), _stream()))
    _count()
    return out


def adaln(x: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor, *, eps: float = 1e-6,
          shift1: Optional[torch.Tensor] = None, scale1: Optional[torch.Tensor] = None, seg_period: int = 0,
          seg_split: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(1 + scale[b]) * LayerNorm(x) + shift[b] on [rows, C]; shift/scale are [B, C] views (row stride free, shared)
    of the Modulation output; rows of sample b are [b*seg_period, (b+1)*seg_period), the first seg_split of them use
    (shift, scale), the rest (shift1, scale1)."""
    _rowmajor2d(x, "x")
    assert x.is_contiguous()
    rows, Cc = x.shape
    if out is None:
        out = torch.empty_like(x)
    assert out.is_contiguous() and out.shape == x.shape
    ld = shift.stride(0)
    for t in (shift, scale, shift1, scale1):
        assert t is None or (t.stride(-1) == 1 and t.stride(0) == ld and t.shape[1] == Cc)
    if seg_period <= 0:
        assert rows % shift.shape[0] == 0
        seg_period = rows // shift.shape[0]
        seg_split = seg_period
    with _prof("adaln", 0.0, 4.0 * rows * Cc):
        _l.check(_l.load().b200_adaln(x.data_ptr(), out.data_ptr(), rows, Cc, eps, shift.data_ptr(), scale.data_ptr(),
                                      _p(shift1), _p(scale1), ld, seg_period, seg_split, _dt(x), _stream()))
    _count()
    return out


def rmsnorm_rows(x: torch.Tensor, scale: torch.Tensor, eps: float = 1e-6, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x * rsqrt(mean(x^2) + eps) * scale over the rows of a contiguous [rows, C] matrix."""
    assert x.dim() == 2 and x.is_contiguous() and scale.is_contiguous() and scale.numel() == x.shape[1]
    if out is None:
        out = torch.empty_like(x)
    with _prof("rmsnorm_rows", 0.0, 4.0 * x.numel()):
        _l.check(_l.load().b200_rmsnorm_rows(x.data_ptr(), scale.data_ptr(), out.data_ptr(), x.shape[0], x.shape[1], eps,
                                             _dt(x), _stream()))
    _count()
    return out


def qk_norm_rope_(qkv: torch.Tensor, heads: int, q_scale: torch.Tensor, k_scale: torch.Tensor, cos: torch.Tensor,
                  sin: torch.Tensor, *, q_scale1: Optional[torch.Tensor] = None, k_scale1: Optional[torch.Tensor] = None,
                  seg_split: int = 0, eps: float = 1e-6) -> torch.Tensor:
    """In place on the q and k thirds of qkv [rows, >= 3*heads*128]: RMSNorm * scale, then RoPE with the fp32 tables
    cos/sin [seg_period, 64] indexed by row % seg_period."""
    _rowmajor2d(qkv, "qkv")
    assert cos.dtype == torch.float32 and sin.dtype == torch.float32 and cos.is_contiguous() and sin.is_contiguous()
    assert cos.shape == sin.shape and cos.shape[1] == 64
    rows = qkv.shape[0]
    period = cos.shape[0]
    assert rows % period == 0
    with _prof("qk_norm_rope", 0.0, 4.0 * rows * 2 * heads * 128):
        _l.check(_l.load().b200_qk_norm_rope(qkv.data_ptr(), rows, heads, 128, qkv.stride(0), q_scale.data_ptr(),
                                             k_scale.data_ptr(), _p(q_scale1), _p(k_scale1), cos.data_ptr(), sin.data_ptr(),
                                             period, seg_split if q_scale1 is not None else period, eps, _dt(qkv), _stream()))
    _count()
    return qkv


def flux_patchify(x: torch.Tensor, dtype: torch.dtype, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x NCHW [B, C, H, W] (fp32 or `dtype`) -> tokens [B*(H/2)*(W/2), 4C] in `dtype`."""
    assert x.is_contiguous() and x.dim() == 4 and x.dtype in (torch.float32, dtype)
    B, Cc, H, W = x.shape
    if out is None:
        out = torch.empty((B * (H // 2) * (W // 2), 4 * Cc), dtype=dtype, device=x.device)
    _rowmajor2d(out, "out")
    with _prof("flux_patchify", 0.0, x.numel() * (x.element_size() + 2.0)):
        _l.check(_l.load().b200_flux_patchify(x.data_ptr(), out.data_ptr(), B, Cc, H, W, out.stride(0),
                                              1 if x.dtype == torch.float32 else 0, _dt(out), _stream()))
    _count()
    return out


def flux_unpatchify(tokens: torch.Tensor, B: int, Cc: int, H: int, W: int, *, nchw_f32: bool,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """tokens [B*(H/2)*(W/2), >= 4C] -> NCHW fp32 [B, C, H, W] (nchw_f32) or NHWC [B, H, W, C] in the tokens' dtype."""
    _rowmajor2d(tokens, "tokens")
    if out is None:
        out = (torch.empty((B, Cc, H, W), dtype=torch.float32, device=tokens.device) if nchw_f32
               else torch.empty((B, H, W, Cc), dtype=tokens.dtype, device=tokens.device))
    assert out.is_contiguous()
    with _prof("flux_unpatchify", 0.0, B * Cc * H * W * (2.0 + out.element_size())):
        _l.check(_l.load().b200_flux_unpatchify(tokens.data_ptr(), out.data_ptr(), B, Cc, H, W, tokens.stride(0),
                                                1 if nchw_f32 else 0, _dt(tokens), _stream()))
    _count()
    return out


def sampler_step(x: torch.Tensor, eps: torch.Tensor, denoised: torch.Tensor, *, kind: int, sigma: float,
                 cfg_scale: float, has_uncond: bool, dt: float = 0.0, noise: Optional[torch.Tensor] = None,
                 noise_scale: float = 0.0, old_denoised: Optional[torch.Tensor] = None, c_x: float = 0.0,
                 c_d: float = 0.0, c_old: float = 0.0, prediction: int = 0) -> None:
    """In-place fused CFG + sampler update; eps is NHWC [(2|1)*B, H, W, ld] (uncond rows first)."""
    assert x.dtype == torch.float32 and x.is_contiguous() and denoised.is_contiguous()
    b, c, h, w = x.shape
    assert eps.is_contiguous() and eps.shape[0] == (2 * b if has_uncond else b)
    d = _l.StepDesc()
    d.kind, d.B, d.C, d.H, d.W = kind, b, c, h, w
    d.ld_eps = eps.shape[-1]
    d.has_uncond = 1 if has_uncond else 0
    d.prediction = prediction
    d.sigma, d.cfg_scale, d.dt, d.noise_scale = sigma, cfg_scale, dt, noise_scale
    d.c_x, d.c_d, d.c_old = c_x, c_d, c_old
    d.eps_dtype = _dt(eps)
    _l.check(_l.load().b200_sampler_step(x.data_ptr(), eps.data_ptr(), _p(noise), denoised.data_ptr(),
                                         _p(old_denoised), C.byref(d), _stream()))
    _count()


def vae_postprocess(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """NHWC [B,H,W,ld>=3] -> fp32 NHWC [B,H,W,3] clamp((x+1)/2, 0, 1)."""
    assert x.dim() == 4 and x.is_contiguous()
    n, h, w, ld = x.shape
    if out is None:
        out = torch.empty((n, h, w, 3), dtype=torch.float32, device=x.device)
    _l.check(_l.load().b200_vae_postprocess(x.data_ptr(), out.data_ptr(), n * h * w, ld, _dt(x), _stream()))
    _count()
    return out


def tile_blend_(acc: torch.Tensor, tile: torch.Tensor, y0: int, x0: int, *, feather: int, bias: float = 0.0) -> torch.Tensor:
    """acc [H, W, 4] fp32 += feather-masked tile NHWC [1, th, tw, ld] (+ bias) at (y0, x0); channel 3 of acc sums the mask."""
    assert acc.dtype == torch.float32 and acc.is_contiguous() and acc.dim() == 3 and acc.shape[2] == 4
    assert tile.is_contiguous() and tile.dim() == 4 and tile.shape[0] == 1
    _, th, tw, ld = tile.shape
    _l.check(_l.load().b200_tile_blend(tile.data_ptr(), acc.data_ptr(), acc.shape[0], acc.shape[1], y0, x0, th, tw, ld, bias,
                                       feather, _dt(tile), _stream()))
    _count()
    return acc


def tile_resolve_(acc: torch.Tensor, out: torch.Tensor, *, accumulate: bool, finalize: bool, final_scale: float = 1.0) -> torch.Tensor:
    """out [H, W, 3] fp32 (+)= acc.rgb / acc.mask; `finalize`: out = clamp(out * final_scale, 0, 1)."""
    assert acc.dtype == torch.float32 and acc.is_contiguous() and out.dtype == torch.float32 and out.is_contiguous()
    assert out.shape == (acc.shape[0], acc.shape[1], 3)
    _l.check(_l.load().b200_tile_resolve(acc.data_ptr(), out.data_ptr(), acc.shape[0] * acc.shape[1], 1 if accumulate else 0,
                                         final_scale, 1 if finalize else 0, _stream()))
    _count()
    return out


def images_to_u8(img: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp32 images in [0, 1] (any shape, contiguous) -> uint8 with the host conversion of modules/processing.py:1039-1040."""
    assert img.dtype == torch.float32 and img.is_contiguous() and img.numel() % 4 == 0
    if out is None:
        out = torch.empty(img.shape, dtype=torch.uint8, device=img.device)
    _l.check(_l.load().b200_images_to_u8(img.data_ptr(), out.data_ptr(), img.numel(), _stream()))
    _count()
    return out


def add_control_(h: torch.Tensor, ctrl: torch.Tensor, *, nhwc: bool = False) -> torch.Tensor:
    """h NHWC [N,H,W,C] += ctrl, in place: ctrl NCHW [N|1,C,H,W] or (nhwc) NHWC [N|1,H,W,C], h.dtype or fp32; a batch-1
    residual is added to every image."""
    assert h.dim() == 4 and h.is_contiguous() and ctrl.is_contiguous()
    n, hh, ww, c = h.shape
    nc = ctrl.shape[0]
    assert nc in (n, 1) and tuple(ctrl.shape[1:]) == ((hh, ww, c) if nhwc else (c, hh, ww)), (tuple(h.shape), tuple(ctrl.shape))
    assert ctrl.dtype in (h.dtype, torch.float32)
    _l.check(_l.load().b200_add_control(h.data_ptr(), ctrl.data_ptr(), n, c, hh, ww, nc, 1 if nhwc else 0,
                                        1 if ctrl.dtype == torch.float32 else 0, _dt(h), _stream()))
    _count()
    return h


def add_nchw_(h: torch.Tensor, ctrl: torch.Tensor) -> torch.Tensor:
    """h NHWC [N,H,W,C] += ctrl NCHW [N|1,C,H,W] (same dtype as h, or fp32), in place."""
    return add_control_(h, ctrl)


def vae_preprocess(pixels: torch.Tensor, dtype: torch.dtype, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """pixels NHWC fp32 [B,H,W,3] in [0,1] -> NHWC [B,H,W,8] in dtype: channels 0-2 = 2x-1, the rest zero."""
    assert pixels.dtype == torch.float32 and pixels.is_contiguous() and pixels.dim() == 4 and pixels.shape[3] == 3
    n, h, w, _ = pixels.shape
    if out is None:
        out = torch.empty((n, h, w, 8), dtype=dtype, device=pixels.device)
    _l.check(_l.load().b200_vae_preprocess(pixels.data_ptr(), out.data_ptr(), n * h * w, _dt(out), _stream()))
    _count()
    return out


def vae_posterior(moments: torch.Tensor, channels: int, noise: Optional[torch.Tensor] = None, scale: float = 1.0,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """moments NHWC [B,h,w,ld>=2C] -> latent NCHW fp32 [B,C,h,w] = (mean + std*noise)*scale (noise None: the mode)."""
    assert moments.dim() == 4 and moments.is_contiguous()
    n, h, w, ld = moments.shape
    if out is None:
        out = torch.empty((n, channels, h, w), dtype=torch.float32, device=moments.device)
    if noise is not None:
        assert noise.dtype == torch.float32 and noise.is_contiguous() and noise.shape == out.shape
    _l.check(_l.load().b200_vae_posterior(moments.data_ptr(), _p(noise), out.data_ptr(), n, channels, h * w, ld, scale,
                                          _dt(moments), _stream()))
    _count()
    return out


def sampler_update(x: torch.Tensor, denoised: torch.Tensor, *, kind: int, sigma: float, dt: float = 0.0,
                   noise: Optional[torch.Tensor] = None, noise_scale: float = 0.0,
                   old_denoised: Optional[torch.Tensor] = None, c_x: float = 0.0, c_d: float = 0.0,
                   c_old: float = 0.0) -> None:
    """In-place sampler update from an already CFG-combined `denoised` (fp32, same shape as x).
    `noise` / `old_denoised` come from the caller's world (Forge's or a user's noise_sampler): anything that is not an fp32
    contiguous tensor of x's shape on x's device is brought there first (broadcast shapes are expanded) — the kernel reads
    raw pointers."""
    assert x.dtype == torch.float32 and x.is_contiguous() and x.is_cuda

    def like_x(t, name):
        if t is None:
            return None
        if not torch.is_tensor(t):
            raise TypeError(f"sampler_update: {name} must be a tensor")
        if t.device != x.device or t.dtype != torch.float32:
            t = t.to(device=x.device, dtype=torch.float32)
        if t.shape != x.shape:
            t = t.expand_as(x)  # raises on shapes that do not broadcast
        return t.contiguous()

    denoised_c = like_x(denoised, "denoised")
    noise = like_x(noise, "noise")
    old_c = like_x(old_denoised, "old_denoised")
    if kind == STEP_DPMPP_2M and old_denoised is not None and old_c.data_ptr() != old_denoised.data_ptr():
        raise ValueError("sampler_update: DPM++ 2M updates old_denoised in place — it must be an fp32 contiguous tensor like x")
    b, c, h, w = x.shape
    d = _l.StepDesc()
    d.kind, d.B, d.C, d.H, d.W = kind, b, c, h, w
    d.sigma, d.dt, d.noise_scale = sigma, dt, noise_scale
    d.c_x, d.c_d, d.c_old = c_x, c_d, c_old
    with torch.cuda.device(x.device):  # the launch goes to x's device whatever the caller's current device is
        _l.check(_l.load().b200_sampler_update(x.data_ptr(), denoised_c.data_ptr(), _p(noise), _p(old_c), C.byref(d),
                                               _stream()))
    _count()


def eps_to_denoised(x: torch.Tensor, eps: torch.Tensor, sigma: torch.Tensor, prediction: int = 0,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x fp32 NCHW [N,C,H,W], eps NHWC [N,H,W,ld] (fp16/bf16), sigma fp32 [N] -> denoised fp32 NCHW."""
    assert x.dtype == torch.float32 and x.is_contiguous() and eps.is_contiguous() and sigma.dtype == torch.float32
    n, c, h, w = x.shape
    if out is None:
        out = torch.empty_like(x)
    _l.check(_l.load().b200_eps_to_denoised(x.data_ptr(), eps.data_ptr(), sigma.data_ptr(), out.data_ptr(), n, c, h, w,
                                            eps.shape[-1], prediction, _dt(eps), _stream()))
    _count()
    return out
