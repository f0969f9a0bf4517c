"""CPU tests of the host-side logic: C-ABI surface, plug-in binding, sampler plans, request sharding (gloo, 2 ranks)."""
import os
import re
import sys
import types

import pytest
import torch

from oracle import sampling as S
from tests.util import assert_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from b200forge import lib
    hdr = open(os.path.join(ROOT, "include", "b200forge.h")).read()
    declared = set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    L = lib.load()  # binds argtypes for every entry of SIGNATURES; AttributeError if a symbol is missing
    for name in declared:
        assert hasattr(L, name), f"{name} declared in b200forge.h but not exported"
    assert declared == set(lib.SIGNATURES), (declared ^ set(lib.SIGNATURES))
    assert L.b200_version() >= 100
    assert isinstance(L.b200_last_error(), bytes)


def test_no_gpu_calls_fail_loudly():
    from b200forge import lib, ops
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert lib.load().b200_device_ok() != 0
    with pytest.raises(Exception):
        ops.gemm(torch.zeros(8, 8, dtype=torch.float16), torch.zeros(8, 8, dtype=torch.float16))


def test_sampler_plans_match_oracle_scalars():
    from b200forge import sampling as BS
    pred = BS.Prediction()
    op = S.EpsPrediction()
    assert torch.equal(pred.sigmas, op.sigmas) and torch.equal(pred.log_sigmas, op.log_sigmas)
    assert torch.equal(BS.get_sigmas_uniform(pred, 30), S.get_sigmas_uniform(op, 30))
    assert torch.equal(BS.get_sigmas_karras(30, pred.sigma_min, pred.sigma_max),
                       S.get_sigmas_karras(30, float(op.sigma_min), float(op.sigma_max)))
    sig = BS.get_sigmas_uniform(pred, 12)
    for st, (a, b) in zip(BS.plan_euler_ancestral(sig), zip(sig[:-1], sig[1:])):
        sd, su = S.get_ancestral_step(float(a), float(b), 1.0)
        assert abs(st.dt - (sd - float(a))) <= 2e-6 * max(1.0, abs(st.dt))
        assert abs(st.noise_scale - (su if float(b) > 0 else 0.0)) <= 2e-6 * max(1.0, su)
    sk = BS.get_sigmas_karras(12, pred.sigma_min, pred.sigma_max)
    plan = BS.plan_dpmpp_2m(sk)
    for i, st in enumerate(plan):
        cx, cd, co = S.dpmpp_2m_coeffs(float(sk[i - 1]) if i > 0 else None, float(sk[i]), float(sk[i + 1]), has_old=i > 0)
        for got, ref in ((st.c_x, cx), (st.c_d, cd), (st.c_old, co)):
            assert abs(got - ref) <= 1e-5 * max(1.0, abs(ref)), (i, got, ref)
    ts = pred.timestep(sig[:-1])
    assert torch.equal(ts, op.timestep(sig[:-1]))


def test_fast_path_predicate():
    from b200forge import plugin
    ctx = torch.zeros(2, 77, 8)
    assert plugin.fast_path_ok({"c_crossattn": ctx, "transformer_options": {}})
    assert plugin.fast_path_ok({"c_crossattn": ctx, "transformer_options": {"patches": {}, "cond_or_uncond": [1, 0]}})
    assert not plugin.fast_path_ok({"c_crossattn": ctx, "transformer_options": {"patches": {"attn1_patch": [lambda *a: a]}}})
    assert not plugin.fast_path_ok({"c_crossattn": ctx, "transformer_options": {"block_modifiers": [lambda *a: a]}})
    assert not plugin.fast_path_ok({"c_crossattn": ctx, "control": object(), "transformer_options": {}})
    assert not plugin.fast_path_ok({"transformer_options": {}})


def _fake_forge_modules():
    ba = types.ModuleType("backend.attention")
    ba.attention_function = lambda q, k, v, heads, mask=None, attn_precision=None, skip_reshape=False: ("ref", q.shape)
    ba.attention_function_single_head_spatial = lambda q, k, v: ("ref1", q.shape)
    un = types.ModuleType("backend.nn.unet")
    un.attention_function = ba.attention_function
    va = types.ModuleType("backend.nn.vae")
    va.attention_function_single_head_spatial = ba.attention_function_single_head_spatial
    ks = types.ModuleType("k_diffusion.sampling")
    ks.sample_euler = lambda *a, **k: "ref_euler"
    ks.sample_euler_ancestral = lambda *a, **k: "ref_euler_a"
    ks.sample_dpmpp_2m = lambda *a, **k: "ref_dpmpp"
    return {"backend.attention": ba, "backend.nn.unet": un, "backend.nn.vae": va, "k_diffusion.sampling": ks}


def test_plugin_rebinds_and_restores_attention():
    from b200forge import attention as A
    from b200forge import plugin
    mods = _fake_forge_modules()
    orig = mods["backend.attention"].attention_function
    plugin.install_attention(mods)
    try:
        assert mods["backend.attention"].attention_function is A.attention_function
        assert mods["backend.nn.unet"].attention_function is A.attention_function  # imported-by-value copy rebound too
        assert mods["backend.nn.vae"].attention_function_single_head_spatial is A.attention_function_single_head_spatial
        # a CPU fp32 call is outside the fused path -> handed to the reference function, not emulated
        q = torch.zeros(1, 4, 64)
        assert A.attention_function(q, q, q, 1) == ("ref", q.shape)
        assert A.attention_function(q.half(), q.half(), q.half(), 1, mask=torch.zeros(4, 4)) == ("ref", q.shape)
    finally:
        plugin.uninstall_attention(mods)
    assert mods["backend.attention"].attention_function is orig and mods["backend.nn.unet"].attention_function is orig
    from b200forge.lib import B200Error
    with pytest.raises(B200Error):  # standalone: no reference to defer to -> loud error
        A.attention_function(torch.zeros(1, 4, 64), torch.zeros(1, 4, 64), torch.zeros(1, 4, 64), 1)


def test_plugin_installs_samplers_and_defers_unsupported_cases():
    from b200forge import k_samplers, plugin
    mods = _fake_forge_modules()
    plugin.install_samplers(mods)
    ks = mods["k_diffusion.sampling"]
    assert ks.sample_euler is k_samplers.sample_euler and ks.sample_dpmpp_2m is k_samplers.sample_dpmpp_2m
    x = torch.zeros(1, 4, 8, 8)  # CPU latent: not the fused path
    assert ks.sample_euler(None, x, torch.tensor([1.0, 0.0])) == "ref_euler"
    assert ks.sample_euler_ancestral(None, x, torch.tensor([1.0, 0.0])) == "ref_euler_a"
    assert ks.sample_dpmpp_2m(None, x, torch.tensor([1.0, 0.0])) == "ref_dpmpp"


def test_plugin_binds_into_the_real_reference_modules(monkeypatch):
    """The modules that import attention_function by value in the reference (recorded in tests/golden/plugin_calls.pt):
    after install() every one of them resolves to the B200 functions, and CPU calls (outside the fused path) still produce
    the reference's own results."""
    from b200forge import attention as A
    from b200forge import plugin
    from oracle import ops as O
    from oracle.golden import load_golden
    g = load_golden("plugin_calls.pt")

    def attention_pytorch(q, k, v, heads, mask=None, attn_precision=None, skip_reshape=False):
        return O.attention(q, k, v, heads)

    def attention_pytorch_single_head_spatial(q, k, v):
        raise AssertionError("not called here")

    for name in ["backend.attention"] + g["attention_importers"] + g["single_head_importers"]:
        monkeypatch.setitem(sys.modules, name, types.ModuleType(name))
    for name in ["backend.attention"] + g["attention_importers"]:
        sys.modules[name].attention_function = attention_pytorch
    for name in ["backend.attention"] + g["single_head_importers"]:
        sys.modules[name].attention_function_single_head_spatial = attention_pytorch_single_head_spatial
    plugin.install_attention()
    try:
        assert all(sys.modules[n].attention_function is A.attention_function for n in ["backend.attention"] + g["attention_importers"])
        assert all(sys.modules[n].attention_function_single_head_spatial is A.attention_function_single_head_spatial
                   for n in ["backend.attention"] + g["single_head_importers"])
        q = g["deferred_q"]
        out = sys.modules["backend.nn.unet"].attention_function(q, q, q, 2)
        assert_close("deferred attention == reference", out, g["deferred_out"], max_abs=1e-5)
    finally:
        plugin.uninstall_attention()
    assert sys.modules["backend.nn.unet"].attention_function.__name__ == g["attention_function_name"] == "attention_pytorch"


def test_operations_class_surface_and_cpu_deferral():
    from b200forge.operations import B200Operations
    for name in ("Linear", "Conv1d", "Conv2d", "Conv3d", "ConvTranspose1d", "ConvTranspose2d", "ConvTranspose3d",
                 "GroupNorm", "LayerNorm", "Embedding"):  # backend/operations.py:455
        assert hasattr(B200Operations, name)
    lin = B200Operations.Linear(16, 8)
    ref = torch.nn.Linear(16, 8)
    ref.load_state_dict(lin.state_dict())
    x = torch.randn(3, 16)
    assert torch.equal(lin(x), ref(x))  # fp32 CPU input: stock torch module semantics
    conv = B200Operations.Conv2d(8, 8, 3, padding=1)
    assert conv(torch.randn(1, 8, 4, 4)).shape == (1, 8, 4, 4)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    from b200forge import dist as D
    seeds = D.shard_seeds(1000, 4, rank, world)
    img = torch.tensor(seeds, dtype=torch.float32).view(4, 1, 1, 1).expand(4, 2, 2, 3).contiguous()
    out = D.gather_to_rank0(img)
    if rank == 0:
        q.put((seeds, out[:, 0, 0, 0].tolist()))
    else:
        assert out is None
        q.put((seeds, None))
    dist.barrier()
    dist.destroy_process_group()


def test_request_sharding_and_gather_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 1000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    gathered = [r[1] for r in res if r[1] is not None][0]
    assert gathered == [1000.0 + i for i in range(8)]  # contiguous-by-seed, independent of the number of ranks
    assert sorted(sum((r[0] for r in res), [])) == list(range(1000, 1008))


def test_flux_schedule_matches_oracle_and_known_values():
    """Product FluxPrediction / Simple scheduler vs the oracle restatement, plus closed-form anchors: mu(4096) = 1.15,
    mu(256) = 0.5, sigma table ends at exactly 1, time_shift(mu, t=0.5) = e^mu / (e^mu + 1)."""
    import math

    import torch

    from b200forge import sampling as S
    from oracle import sampling as OS
    p = S.FluxPrediction()
    assert abs(p.mu - 1.15) < 1e-12 and abs(S.FluxPrediction(seq_len=256).mu - 0.5) < 1e-12
    assert abs(OS.flux_calculate_shift(1024) - (0.5 + (1.15 - 0.5) * (1024 - 256) / (4096 - 256))) < 1e-12
    assert torch.equal(p.sigmas, OS.flux_sigma_table()) and float(p.sigmas[-1]) == 1.0
    assert abs(float(p.sigmas[4999]) - math.exp(1.15) / (math.exp(1.15) + 1.0)) < 1e-6
    for n in (4, 20, 28):
        a, b = S.get_sigmas_simple(p.sigmas, n), OS.simple_scheduler(n, OS.flux_sigma_table())
        assert torch.equal(a, b) and float(a[0]) == 1.0 and float(a[-1]) == 0.0 and bool((a[:-1] > a[1:]).all())
    noise = torch.randn(2, 16, 4, 4)
    assert torch.equal(p.noise_scaling(1.0, noise), OS.const_noise_scaling(1.0, noise, torch.zeros_like(noise)))


def test_img2img_schedule_matches_setup_img2img_steps():
    """modules/sd_samplers_common.py:24-33 (default options) + the sigma slice of sample_img2img
    (modules/sd_samplers_kdiffusion.py:140-143): t_enc = int(min(strength, 0.999) * steps), last t_enc + 2 sigmas."""
    import torch

    from b200forge.pipeline import Txt2ImgPipeline
    sig = torch.linspace(14.6, 0.03, 30).tolist() + [0.0]
    sig = torch.tensor(sig)
    for steps, strength, t_enc in ((30, 0.75, 22), (30, 1.0, 29), (30, 0.05, 1), (30, 0.0, 0), (20, 0.5, 10)):
        s = Txt2ImgPipeline.img2img_schedule(sig[: steps + 1] if steps == 30 else torch.cat([sig[:steps], sig[-1:]]), steps, strength)
        assert len(s) == t_enc + 2, (steps, strength, len(s))
        assert float(s[-1]) == 0.0


def test_ctypes_descriptors_match_the_c_header_layout(tmp_path):
    """The ctypes Structures in lib.py must have exactly the size and field offsets of the structs in
    include/b200forge.h: a tiny C program (gcc) prints sizeof / offsetof for every field."""
    import ctypes as C
    import os
    import subprocess

    from b200forge import lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pairs = {"b200_gemm_desc": lib.GemmDesc, "b200_conv3x3_desc": lib.Conv3x3Desc, "b200_attn_desc": lib.AttnDesc,
             "b200_gn_desc": lib.GnDesc, "b200_step_desc": lib.StepDesc}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "b200forge.h"', 'int main(void) {']
    for cname, cls in pairs.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    seen = 0
    for ln in out:
        if not ln:
            continue
        cname, field, val = ln.split()
        cls = pairs[cname]
        if field == "size":
            assert C.sizeof(cls) == int(val), (cname, C.sizeof(cls), val)
        else:
            assert getattr(cls, field).offset == int(val), (cname, field, getattr(cls, field).offset, val)
        seen += 1
    assert seen == sum(len(c._fields_) + 1 for c in pairs.values())


def test_supported_latent_sizes_and_deferral():
    """The TMA convolution path tiles power-of-two (<= 128) and multiple-of-128 widths; the engines report what they
    support and the P3 / P5 wrappers hand everything else back to Forge's own callables."""
    import torch

    from b200forge import ops, plugin
    assert all(ops.conv3x3_supported(s, s) for s in (1, 2, 4, 8, 16, 32, 64, 128, 256, 1024))
    assert ops.conv3x3_supported(64, 128) and ops.conv3x3_supported(128, 256)
    assert not any(ops.conv3x3_supported(h, w) for h, w in ((104, 152), (112, 144), (96, 168), (80, 192 + 8)))

    class Eng:  # stands in for UNetEngine: the wrapper must not touch it for an unsupported size
        has_label = False

        def supports_latent(self, h, w):
            return ops.conv3x3_supported(h, w)

    class P:
        prediction_type = "epsilon"

    w = plugin.UNetWrapper(Eng(), P())
    sentinel = torch.zeros(1)
    x = torch.zeros(2, 4, 104, 152)
    out = w(lambda xx, ss, **kw: sentinel, {"input": x, "timestep": torch.ones(2), "c": {"c_crossattn": torch.zeros(2, 77, 8)}})
    assert out is sentinel and w.calls_reference == 1


def _emulated_sampler_update(x, denoised, *, kind, sigma, dt=0.0, noise=None, noise_scale=0.0, old_denoised=None,
                             c_x=0.0, c_d=0.0, c_old=0.0):
    """fp32 torch restatement of csrc/sampler.cu::sampler_update_kernel (the three step kinds), so that the host logic
    of k_samplers.py can be pinned against the reference's loops without a GPU.  The kernel itself is compared with the
    oracle in tests/test_kernels_gpu.py / test_plugin_gpu.py."""
    import torch

    from b200forge import ops
    f = torch.float32
    if kind == ops.STEP_EULER:
        xn = x + ((x - denoised) / torch.tensor(sigma, dtype=f)) * torch.tensor(dt, dtype=f)
        if noise_scale != 0.0:
            xn = xn + noise * torch.tensor(noise_scale, dtype=f)
    else:
        xn = torch.tensor(c_x, dtype=f) * x + torch.tensor(c_d, dtype=f) * denoised
        if c_old != 0.0:
            xn = xn + torch.tensor(c_old, dtype=f) * old_denoised
        if kind == ops.STEP_LINEAR:
            if noise_scale != 0.0:
                xn = xn + torch.tensor(noise_scale, dtype=f) * noise
        else:
            old_denoised.copy_(denoised)
    x.copy_(xn)


@pytest.mark.parametrize("key", ["sample_heun", "sample_dpm_2", "sample_dpm_2_ancestral", "sample_dpmpp_2s_ancestral",
                                 "sample_lms", "sample_dpmpp_sde", "sample_dpmpp_2m_sde", "sample_dpmpp_2m_sde_heun",
                                 "sample_dpmpp_3m_sde", "sample_heunpp2", "sample_ipndm", "sample_ipndm_v", "sample_deis"])
def test_k_sampler_host_logic_vs_reference_golden(key, monkeypatch):
    """The per-step coefficient plans of the fused samplers (k_samplers.py) drive an emulation of the update kernel on the
    CPU and must land on the reference's k-diffusion result for the same toy denoiser and noise stream
    (tests/golden/samplers_toy.pt, made by oracle/gen_golden.py from k_diffusion/sampling.py itself)."""
    import os

    import torch

    from b200forge import k_samplers
    from oracle import sampling as OS
    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "samplers_toy.pt"), weights_only=False)
    monkeypatch.setattr(k_samplers.ops, "sampler_update", _emulated_sampler_update)
    monkeypatch.setattr(k_samplers, "_fusable", lambda x: True)
    name = key.replace("_heun", "") if key.endswith("sde_heun") else key
    kw = {"solver_type": "heun"} if key.endswith("sde_heun") else {}
    k = iter(range(g["noise"].shape[0]))
    if "ancestral" in name or "sde" in name:
        kw["noise_sampler"] = lambda s, sn: g["noise"][next(k)]
    seen = []
    out = getattr(k_samplers, name)(lambda x, sigma, **kwargs: OS.toy_denoiser(x, sigma), g["x0"].clone(), g["sigmas"],
                                    extra_args={}, callback=lambda d: seen.append(d["i"]), disable=True, **kw)
    assert seen == list(range(len(g["sigmas"]) - 1))
    err = (out - g[key]).abs().max().item()
    scale = g[key].abs().max().item()
    assert err <= 2e-5 * max(1.0, scale), (key, err, scale)


@pytest.mark.parametrize("name", ["sample_euler_ancestral", "sample_dpm_2_ancestral"])
def test_rectified_flow_ancestral_samplers_vs_reference_golden(name, monkeypatch):
    """For a Flux model the reference's Euler a / DPM2 a switch to their rectified-flow variants
    (k_diffusion/sampling.py:143-144, 162-186, 251-252, 278-309); the fused versions dispatch the same way.  The dispatch is
    on the predictor's type, backend.modules.k_prediction.PredictionFlux, stood in for here by a class of that name."""
    import os

    import torch

    k_prediction = types.ModuleType("backend.modules.k_prediction")

    class PredictionFlux:
        prediction_type = "const"

    k_prediction.PredictionFlux = PredictionFlux
    monkeypatch.setitem(sys.modules, "backend.modules.k_prediction", k_prediction)

    from b200forge import k_samplers
    from oracle import sampling as OS
    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "samplers_toy.pt"), weights_only=False)
    monkeypatch.setattr(k_samplers.ops, "sampler_update", _emulated_sampler_update)
    monkeypatch.setattr(k_samplers, "_fusable", lambda x: True)

    class FluxModel:
        class _Inner:
            predictor = PredictionFlux()
        inner_model = _Inner()

        def __call__(self, x, sigma, **kw):
            return OS.toy_denoiser(x, sigma)

    k = iter(range(g["noise"].shape[0]))
    out = getattr(k_samplers, name)(FluxModel(), g["flux_x0"].clone(), g["flux_sigmas"], extra_args={}, disable=True,
                                    noise_sampler=lambda s, sn: g["noise"][next(k)])
    err = (out - g[name + "_rf"]).abs().max().item()
    assert err <= 2e-5 * max(1.0, g[name + "_rf"].abs().max().item()), (name, err)


def test_restart_and_lcm_sampler_host_logic(monkeypatch):
    """Restart (modules/sd_samplers_extra.py:7-74) against the reference file's own output around the toy denoiser, with the
    re-noising draws replayed through k-diffusion's torch handle; LCM (modules/sd_samplers_lcm.py:68-82 — that module needs
    Forge's `modules.shared`, so its ten-line loop is pinned against its restatement here, not against an import)."""
    import os
    import sys
    import types

    import torch

    from b200forge import k_samplers
    from oracle import sampling as OS
    g = torch.load(os.path.join(os.path.dirname(__file__), "golden", "samplers_toy.pt"), weights_only=False)
    monkeypatch.setattr(k_samplers.ops, "sampler_update", _emulated_sampler_update)
    monkeypatch.setattr(k_samplers, "_fusable", lambda x: True)
    draws = iter(range(g["restart_noise"].shape[0]))
    fake_t = types.SimpleNamespace(randn_like=lambda x: g["restart_noise"][next(draws)])
    monkeypatch.setitem(sys.modules, "k_diffusion", types.ModuleType("k_diffusion"))
    ks = types.ModuleType("k_diffusion.sampling")
    ks.torch = fake_t
    monkeypatch.setitem(sys.modules, "k_diffusion.sampling", ks)
    seen = []
    out = k_samplers.restart_sampler(lambda x, sigma, **kw: OS.toy_denoiser(x, sigma), g["restart_x0"].clone(), g["restart_sigmas"],
                                     extra_args={}, callback=lambda d: seen.append(d["i"]), disable=True)
    err = (out - g["restart_sampler"]).abs().max().item()
    assert err <= 3e-5 * max(1.0, g["restart_sampler"].abs().max().item()), err
    assert seen == list(range(len(seen))) and len(seen) > 15 and next(draws) == 1  # one restart jump -> one noise draw
    # LCM
    sig = g["sigmas"]
    noise = g["noise"]
    k = iter(range(noise.shape[0]))
    out = k_samplers.sample_lcm(lambda x, sigma, **kw: OS.toy_denoiser(x, sigma), g["x0"].clone(), sig, extra_args={}, disable=True,
                                noise_sampler=lambda s, sn: noise[next(k)])
    x = g["x0"].clone()
    k = iter(range(noise.shape[0]))
    for i in range(len(sig) - 1):
        x = OS.toy_denoiser(x, sig[i] * x.new_ones([x.shape[0]]))
        if sig[i + 1] > 0:
            x = x + sig[i + 1] * noise[next(k)]
    assert (out - x).abs().max().item() <= 1e-5


def test_upsample_folded_conv_weights_and_emulation():
    """pack_conv3x3_up2x + the parity arithmetic of b200_conv3x3_up2x (as emulated in tests/ops_emulator.py) reproduce
    F.interpolate(nearest, x2) followed by the 3x3 convolution (backend/nn/unet.py:330-355) exactly in fp32, borders and
    odd sizes included."""
    import torch
    import torch.nn.functional as F
    from b200forge import ops
    from tests import ops_emulator as E
    g = torch.Generator().manual_seed(7)
    for (n, h, w, c, co) in [(2, 5, 7, 64, 64), (1, 1, 1, 64, 128), (1, 8, 8, 128, 64)]:
        x = torch.randn(n, c, h, w, generator=g)
        wt = torch.randn(co, c, 3, 3, generator=g) * (9 * c) ** -0.5
        b = torch.randn(co, generator=g)
        w4 = ops.pack_conv3x3_up2x(wt)
        assert w4.shape == (4 * co, 4 * c)
        y = E.conv3x3_up2x(x.permute(0, 2, 3, 1).contiguous(), w4, b)
        ref = F.conv2d(F.interpolate(x, scale_factor=2, mode="nearest"), wt, b, padding=1).permute(0, 2, 3, 1)
        assert y.shape == ref.shape
        assert (y - ref).abs().max().item() < 2e-5
