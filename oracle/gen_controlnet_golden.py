"""ORACLE tooling — generates tests/golden/controlnet_*.pt by running the UNMODIFIED reference ControlNet
(backend.nn.cnets.cldm.ControlNet, imported from the reference tree through oracle/ref_import.py) on CPU in fp32.

    python -m oracle.gen_controlnet_golden     # needs the reference tree

Each fixture holds two calls on the same latent batch: a batch-1 hint (broadcast onto the batch, what Forge passes
for one control image) and a batch-N hint.  Weights come from `oracle.controlnet.random_controlnet_state_dict(cfg,
seed=...)` and the inputs from `oracle.golden.seeded_inputs(shapes, seed)`; only seeds, shapes and outputs are stored.
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import controlnet as OC  # noqa: E402
from oracle import ref_import  # noqa: E402
from oracle.golden import GOLD, seeded_inputs  # noqa: E402

WEIGHT_SEED, INPUT_SEED = 11, 12
LATENT = (16, 8)  # non-square, every level tiles on the TMA convolution path; keeps each fixture under 1 MB


def input_shapes(cfg: dict, n: int = 2, hw=LATENT) -> dict:
    h, w = hw
    s = {"x": (n, cfg["in_channels"], h, w), "hint1": (1, cfg["hint_channels"], 8 * h, 8 * w),
         "hintN": (n, cfg["hint_channels"], 8 * h, 8 * w), "context": (n, 77, cfg["context_dim"])}
    if cfg.get("adm_in_channels"):
        s["y"] = (n, cfg["adm_in_channels"])
    return s


def make_inputs(shapes: dict, seed: int) -> dict:
    """The fixture's inputs from its stored shapes and seed: N(0,1) latents / context / y, hints in [0, 1)."""
    names = sorted(shapes)
    vals = dict(zip(names, seeded_inputs([shapes[k] for k in names], seed)))
    for k in ("hint1", "hintN"):
        vals[k] = torch.sigmoid(vals[k])
    vals["t"] = torch.tensor([981.0, 23.0])[: shapes["x"][0]]
    return vals


def gen_controlnet(name: str) -> None:
    from backend.nn.cnets.cldm import ControlNet
    cfg = OC.CONFIGS[name]
    sd = OC.random_controlnet_state_dict(cfg, cfg["hint_channels"], seed=WEIGHT_SEED)
    m = ControlNet(**cfg).eval()
    m.load_state_dict(sd, strict=True)
    shapes = input_shapes(cfg)
    v = make_inputs(shapes, INPUT_SEED)
    outs = {}
    with torch.no_grad():
        for k in ("hint1", "hintN"):
            outs[k] = [o.clone() for o in m(x=v["x"], hint=v[k], timesteps=v["t"], context=v["context"], y=v.get("y"))]
    torch.save(dict(config=name, weight_seed=WEIGHT_SEED, input_seed=INPUT_SEED, shapes=shapes, out=outs),
               os.path.join(GOLD, f"controlnet_{name}.pt"))
    print("controlnet", name, [tuple(o.shape) for o in outs["hint1"]], "std", [round(o.std().item(), 3) for o in outs["hint1"]])


if __name__ == "__main__":
    ref_import.load()
    for n in sys.argv[1:] or ["tiny_xl", "tiny_15h"]:
        gen_controlnet(n)
