"""ControlNet engine and the P6 plug point (plugin.ControlNetWrapper) on the CPU: the engine's launch sequence runs over the
torch emulation of the kernel wrappers (tests/ops_emulator.py, plus the control-add op below) and is compared with the
reference's own outputs (tests/golden/controlnet_*.pt, oracle/gen_controlnet_golden.py)."""
from __future__ import annotations

import pytest
import torch

from b200forge import ops, plugin
from b200forge.controlnet_engine import ControlNetEngine, controlnet_config
from oracle import controlnet as OC
from oracle.gen_controlnet_golden import make_inputs
from oracle.golden import load_golden
from tests import ops_emulator
from tests.util import assert_close


def add_control_(h, ctrl, *, nhwc=False):
    """csrc/elementwise.cu::add_control_kernel: h NHWC += ctrl (NCHW or NHWC, batch N or 1), in place."""
    c = ctrl.float() if nhwc else ctrl.float().permute(0, 2, 3, 1)
    assert c.shape[0] in (h.shape[0], 1) and c.shape[1:] == h.shape[1:]
    h.copy_((h.float() + c).to(h.dtype))
    return h


@pytest.fixture(autouse=True)
def _emulated_ops(monkeypatch):
    ops_emulator.install(monkeypatch)
    monkeypatch.setattr(ops, "add_control_", add_control_)


def _case(name):
    g = load_golden(f"controlnet_{name}.pt")
    cfg = OC.CONFIGS[name]
    sd = OC.random_controlnet_state_dict(cfg, cfg["hint_channels"], seed=g["weight_seed"])
    return g, cfg, sd, make_inputs(g["shapes"], g["input_seed"])


@pytest.mark.parametrize("name", ["tiny_xl", "tiny_15h"])
@pytest.mark.parametrize("hint", ["hint1", "hintN"])
def test_oracle_vs_reference_golden(name, hint):
    g, cfg, sd, v = _case(name)
    with torch.no_grad():
        outs = OC.controlnet_forward(sd, cfg, v["x"], v[hint], v["t"], v["context"], v.get("y"))
    assert len(outs) == len(g["out"][hint])
    for i, (o, r) in enumerate(zip(outs, g["out"][hint])):
        assert_close(f"oracle controlnet {name} {hint} out {i}", o, r, max_abs=5e-5)


@pytest.mark.parametrize("name", ["tiny_xl", "tiny_15h"])
@pytest.mark.parametrize("hint", ["hint1", "hintN"])
def test_engine_host_logic_vs_reference_golden(name, hint):
    g, cfg, sd, v = _case(name)
    eng = ControlNetEngine(cfg, sd, dtype=torch.float32, device="cpu")
    outs = eng.forward(v["x"], v[hint], v["t"], v["context"], v.get("y"))
    assert len(outs) == len(g["out"][hint])
    for i, (o, r) in enumerate(zip(outs, g["out"][hint])):
        assert o.is_contiguous() and o.dtype == torch.float32
        assert_close(f"emulated ControlNetEngine {name} {hint} out {i}", o, r, max_abs=3e-4)


class _StandInControlNet:
    """What the P6 wrapper reads from a cldm.ControlNet: the constructor attributes, state_dict(), modules() and the
    call itself (here the oracle)."""

    def __init__(self, cfg, sd):
        self.cfg, self.sd = cfg, sd
        self.model_channels = cfg["model_channels"]
        self.num_res_blocks = list(cfg["num_res_blocks"])
        self.channel_mult = tuple(cfg["channel_mult"])
        self.num_heads, self.num_head_channels = cfg["num_heads"], cfg["num_head_channels"]
        self.calls = 0

    def state_dict(self):
        return dict(self.sd)

    def modules(self):
        return iter([self])

    def __call__(self, x, hint, timesteps, context, y=None):
        self.calls += 1
        return OC.controlnet_forward(self.sd, self.cfg, x.float(), hint.float(), timesteps, context.float(),
                                     None if y is None else y.float())


class _Holder:  # backend.patcher.controlnet.ControlNet: `device` is where get_control's no-wrapper branch moves the hint
    device = torch.device("cpu")


class ControlLora(_Holder):
    pass


@pytest.mark.parametrize("name", ["tiny_xl", "tiny_15h"])
def test_controlnet_config_from_a_module(name):
    _, cfg, sd, _ = _case(name)
    got = controlnet_config(_StandInControlNet(cfg, sd))
    for k in ("in_channels", "model_channels", "channel_mult", "transformer_depth", "transformer_depth_middle", "num_heads",
              "num_head_channels", "use_linear_in_transformer", "context_dim", "adm_in_channels", "num_classes", "hint_channels"):
        assert (list(got[k]) if isinstance(got[k], (list, tuple)) else got[k]) == \
               (list(cfg[k]) if isinstance(cfg[k], (list, tuple)) else cfg[k]), k
    assert list(got["num_res_blocks"]) == list(cfg["num_res_blocks"])


def _args(v, hint, dtype=torch.float16):
    return dict(x=v["x"].to(dtype), hint=hint, timesteps=v["t"], context=v["context"].to(dtype),
                y=None if v.get("y") is None else v["y"].to(dtype))


def test_p6_wrapper_contract(monkeypatch):
    g, cfg, sd, v = _case("tiny_xl")
    monkeypatch.setattr(plugin, "_on_device", lambda t: True)
    inner = _StandInControlNet(cfg, sd)
    w = plugin.ControlNetWrapper()
    hint = v["hint1"].clone()
    a = _args(v, hint)
    outs = w(**a, model=_Holder(), inner_model=inner)
    assert (w.calls_fast, w.calls_reference, inner.calls) == (1, 0, 0)
    assert len(outs) == len(g["out"]["hint1"])
    for i, (o, r) in enumerate(zip(outs, g["out"]["hint1"])):
        assert o.dtype == torch.float16 and o.is_contiguous() and o.shape == r.shape  # NCHW, x's dtype
        assert_close(f"P6 out {i}", o, r, rel_rms=5e-3)
    # fresh tensors: control_merge scales them in place (`x *= strength`), which must not reach the next call
    ref0 = outs[0].clone()
    for o in outs:
        o.mul_(0.0)
    outs2 = w(**a, model=_Holder(), inner_model=inner)
    assert all(o2.data_ptr() != o.data_ptr() for o, o2 in zip(outs, outs2))
    assert torch.equal(outs2[0], ref0)
    assert len(w.engines) == 1
    # a hint edited in place (same tensor, new version) gives a new guided_hint
    hint.mul_(0.5)
    outs3 = w(**a, model=_Holder(), inner_model=inner)
    with torch.no_grad():
        ref3 = OC.controlnet_forward(sd, cfg, v["x"], hint, v["t"], v["context"], v["y"])
    assert not torch.equal(outs3[0], outs2[0])
    for i, (o, r) in enumerate(zip(outs3, ref3)):
        assert_close(f"P6 out {i} after an in-place hint edit", o, r, rel_rms=5e-3)
    assert (w.calls_fast, w.calls_reference, inner.calls) == (3, 0, 0)


def test_p6_wrapper_defers(monkeypatch):
    g, cfg, sd, v = _case("tiny_xl")
    inner = _StandInControlNet(cfg, sd)
    w = plugin.ControlNetWrapper()
    a = _args(v, v["hint1"])
    # CPU tensors: get_control's own branch, inner_model(x=, hint=hint.to(model.device), ...)
    outs = w(**a, model=_Holder(), inner_model=inner)
    ref = inner(**a)
    assert all(torch.equal(o, r) for o, r in zip(outs, ref))
    assert (w.calls_fast, w.calls_reference) == (0, 1)
    monkeypatch.setattr(plugin, "_on_device", lambda t: True)
    # Control-LoRA: by class, or by a layer that carries up / down
    outs = w(**a, model=ControlLora(), inner_model=inner)
    assert all(torch.equal(o, r) for o, r in zip(outs, ref))
    lora_like = _StandInControlNet(cfg, sd)
    lora_like.up, lora_like.down = None, None
    w(**a, model=_Holder(), inner_model=lora_like)
    assert (w.calls_fast, w.calls_reference) == (0, 3)
    # fp32, a hint that is not 8x the latent, B200_CONTROLNET=0
    w(**_args(v, v["hint1"], torch.float32), model=_Holder(), inner_model=inner)
    with pytest.raises(RuntimeError):  # the reference model cannot add a guided hint of the wrong size either
        w(**_args(v, v["hint1"][:, :, ::2, ::2]), model=_Holder(), inner_model=inner)
    monkeypatch.setenv("B200_CONTROLNET", "0")
    w(**a, model=_Holder(), inner_model=inner)
    assert (w.calls_fast, w.calls_reference) == (0, 6)
    # T2I-Adapter: wrapper(hint=, model=, inner_model=, inner_t2i_model=) -> inner_model(hint)
    t2i = lambda h: [h * 2.0]  # noqa: E731
    res = w(hint=v["hint1"], model=_Holder(), inner_model=t2i, inner_t2i_model=t2i)
    assert torch.equal(res[0], v["hint1"] * 2.0)
    assert (w.calls_fast, w.calls_reference) == (0, 7)


def test_unet_control_fits_and_batch1_residuals():
    """P3 with T2I-Adapter residuals of one hint image (batch 1 on a batch-2 latent): accepted and broadcast, like the
    reference's `h += ctrl`; a residual that does not broadcast is handed back to Forge (which skips it with a warning)."""
    from b200forge.unet_engine import UNetEngine
    from oracle import configs as CF
    from oracle import unet as OU
    g = load_golden("unet_tiny_xl_control.pt")
    cfg = CF.CONFIGS["tiny_xl"]
    sd = OU.random_state_dict(cfg, seed=1)
    eng = UNetEngine(cfg, sd, dtype=torch.float32, device="cpu")
    ctrl1 = {k: [None if t is None else t[:1].clone() for t in lst] for k, lst in g["control"].items()}
    n, hh, ww = g["x"].shape[0], g["x"].shape[2], g["x"].shape[3]
    assert eng.control_fits(g["control"], n, hh, ww) and eng.control_fits(ctrl1, n, hh, ww)
    out = eng.forward(g["x"], g["t"], g["context"], g["y"], control=ctrl1)
    with torch.no_grad():
        ref = OU.unet_forward(sd, cfg, g["x"], g["t"], g["context"], g["y"], control=ctrl1)
    assert_close("emulated UNetEngine + batch-1 control vs oracle", out, ref, max_abs=3e-4)
    bad = {k: list(v) for k, v in ctrl1.items()}
    bad["input"][-1] = bad["input"][-1][:, :, :4]
    assert not eng.control_fits(bad, n, hh, ww)
    bad["input"][-1] = torch.zeros((3,) + tuple(ctrl1["input"][-1].shape[1:]))
    assert not eng.control_fits(bad, n, hh, ww)


@pytest.mark.parametrize("name", ["tiny_xl_noattn", "tiny_xl_noattn_nomid"])
def test_controlnet_without_cross_attention(name, monkeypatch):
    """A ControlNet with every transformer depth 0 has no key to read the context width from: its config is still derived
    and the engine serves it (a depth-0 SpatialTransformer is GroupNorm + proj_in + proj_out)."""
    cfg = OC.CONFIGS[name]
    sd = OC.random_controlnet_state_dict(cfg, 3, seed=5)
    assert not any("attn2" in k for k in sd)
    got = controlnet_config(_StandInControlNet(cfg, sd))
    assert got["context_dim"] is None and got["transformer_depth"] == [0] * 6
    assert got["transformer_depth_middle"] == cfg["transformer_depth_middle"]
    monkeypatch.setattr(plugin, "_on_device", lambda t: True)
    inner = _StandInControlNet(cfg, sd)
    w = plugin.ControlNetWrapper()
    g = torch.Generator().manual_seed(6)
    x, hint = torch.randn(2, 4, 16, 8, generator=g), torch.rand(1, 3, 128, 64, generator=g)
    ctx, y, t = torch.randn(2, 77, cfg["context_dim"], generator=g), torch.randn(2, cfg["adm_in_channels"], generator=g), \
        torch.tensor([900.0, 20.0])
    outs = w(x=x.half(), hint=hint, timesteps=t, context=ctx.half(), y=y.half(), model=_Holder(), inner_model=inner)
    assert (w.calls_fast, w.calls_reference) == (1, 0)
    with torch.no_grad():
        ref = OC.controlnet_forward(sd, cfg, x.half().float(), hint, t, ctx.half().float(), y.half().float())
    for i, (o, r) in enumerate(zip(outs, ref)):
        assert_close(f"{name} P6 out {i}", o, r, rel_rms=5e-3)


def test_p6_defers_a_model_the_engine_cannot_be_built_for(monkeypatch):
    """Outside B200_STRICT=1 a model whose engine cannot be built runs in Forge, as it did without the plug point; the
    decision (like the Control-LoRA walk over its modules) is taken once per model."""
    g, cfg, sd, v = _case("tiny_xl")
    monkeypatch.setattr(plugin, "_on_device", lambda t: True)
    broken = _StandInControlNet(cfg, {k: t for k, t in sd.items() if not k.startswith("input_hint_block.4.")})
    walks = []
    broken.modules = lambda: walks.append(1) or iter([broken])
    w = plugin.ControlNetWrapper()
    a = _args(v, v["hint1"])
    with pytest.raises(KeyError):  # the stand-in's own forward needs the weights the engine missed
        w(**a, model=_Holder(), inner_model=broken)
    with pytest.raises(KeyError):
        w(**a, model=_Holder(), inner_model=broken)
    assert (w.calls_fast, w.calls_reference, len(walks)) == (0, 2, 1)
    assert "KeyError" in w.unserved[broken] and broken not in w.engines
    monkeypatch.setenv("B200_STRICT", "1")
    strict = plugin.ControlNetWrapper()
    with pytest.raises(KeyError):  # raised by the engine build, before any call is handed back
        strict(**a, model=_Holder(), inner_model=broken)
    assert strict.calls_reference == 0 and strict.calls_fast == 0
    # a servable model: the module walk runs once, not once per call
    ok = _StandInControlNet(cfg, sd)
    walks.clear()
    ok.modules = lambda: walks.append(1) or iter([ok])
    for _ in range(3):
        w(**a, model=_Holder(), inner_model=ok)
    assert w.calls_fast == 3 and len(walks) == 1
