"""Helpers shared by the golden-vector generator (oracle/gen_golden.py) and the tests that read its fixtures: loading a
fixture, and the seeded tensors a fixture stores only the seed of."""
from __future__ import annotations

import os

import torch

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def control_residuals(shapes: dict, seed: int) -> dict:
    """ControlNet-style residuals, N(0, 0.3^2): one per input block (listed in pop order: block 0 last), one for the middle
    block, one per output skip with a None entry at index 2."""
    g = torch.Generator().manual_seed(seed)
    ins = [torch.randn(tuple(s), generator=g) * 0.3 for s in shapes["input"]]
    return {"input": list(reversed(ins)),                                   # popped from the end: block 0 first
            "middle": [torch.randn(tuple(shapes["middle"][0]), generator=g) * 0.3],
            "output": [None if i == 2 else torch.randn(tuple(s), generator=g) * 0.3 for i, s in enumerate(shapes["input"])]}


def load_golden(name: str) -> dict:
    """torch.load of tests/golden/<name>, with the control residuals of unet_*_control.pt regenerated."""
    g = torch.load(os.path.join(GOLD, name), weights_only=False)
    if "control_seed" in g:
        g["control"] = control_residuals(g["control_shapes"], g["control_seed"])
    return g


def seeded_inputs(shapes, seed):
    """N(0, 1) tensors of the given shapes from one CPU generator (the tests regenerate them from the stored seed)."""
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(tuple(s), generator=g) for s in shapes]


def sample_index(numel, seed, n=512):
    """A fixed, seeded subset of a flattened output's elements (all of them when there are at most n)."""
    if numel <= n:
        return torch.arange(numel)
    return torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:n].sort().values
