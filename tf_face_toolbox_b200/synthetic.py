"""Synthetic embeddings / labels / class weights of the BASELINE.json shapes (SURVEY.md 8d).

Generated on the CPU with fixed seeds so the CPU oracle and the GPU path see identical
bits.  W ~ N(0, 0.01^2) fp32 in the reference layout [D, C] (nets/sphere.py:86), labels
uniform int32 (data.py:259), and X rows a 4-way mixture around the target direction
(x_i = a_i * what_{y_i} * sqrt(D) + N(0, I), a_i in {+1.5,+0.3,-0.3,-1.5} by i mod 4) so that
all four psi branches k = 0..3 are exercised.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import torch

# BASELINE.json configs: name -> (B, D, C, mode)
CONFIGS = {
    "cfg1": dict(B=256, D=512, C=10572, mode="fp32"),
    "cfg2_head": dict(B=512, D=512, C=10572, mode="bf16"),
    "cfg3": dict(B=512, D=512, C=85742, mode="bf16"),
    "cfg4": dict(B=1024, D=512, C=1000000, mode="bf16"),
    "cfg5_head": dict(B=2048, D=512, C=85742, mode="bf16"),
    # config 5 proper: the head plus the center loss (loss.py:29-45) on the same batch
    "cfg5": dict(B=2048, D=512, C=85742, mode="bf16", center=True),
}

MIX = (1.5, 0.3, -0.3, -1.5)


@dataclass
class HeadInputs:
    X: torch.Tensor        # [B, D] fp32
    W: torch.Tensor        # [D, C] fp32
    y: torch.Tensor        # [B] int32


def make_inputs(B: int, D: int, C: int, seed: int = 1234, w_std: float = 0.01,
                labels: Optional[torch.Tensor] = None) -> HeadInputs:
    """`labels` [B] replaces the uniform draw (X is built around the given classes)."""
    gw = torch.Generator().manual_seed(seed)
    gy = torch.Generator().manual_seed(seed + 1)
    gx = torch.Generator().manual_seed(seed + 2)
    W = torch.randn(D, C, generator=gw, dtype=torch.float32) * w_std
    if labels is None:
        y = torch.randint(0, C, (B,), generator=gy, dtype=torch.int64).to(torch.int32)
    else:
        y = labels.to(torch.int32).contiguous()
    wy = W[:, y.long()].t().contiguous()                        # [B, D]
    wy = wy / wy.norm(dim=1, keepdim=True)
    a = torch.tensor(MIX, dtype=torch.float32)[torch.arange(B) % 4]
    X = a[:, None] * wy * math.sqrt(D) + torch.randn(B, D, generator=gx, dtype=torch.float32)
    return HeadInputs(X.contiguous(), W.contiguous(), y)
