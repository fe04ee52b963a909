"""Oracles of VectorQuantizerEMA's codebook update (test infrastructure; never imported by the product path).

Two restatements of the exponential-moving-average codebook update of van den Oord et al. 2017, App. A.1, with the
semantics of the `Quantize` module of rosinality/vq-vae-2-pytorch.  Neither is reference code: the reference trains its
codebook by gradient, and rosinality's module is not vendored here.

- `ema_update_fp64`: the update as the product documents it, in float64.  The arbiter of the GPU tests.
- `rosinality_train_step`: a literal float32 transcription of the training branch of rosinality's `Quantize.forward`
  (one-hot, `flatten.T @ onehot`, `mul_` / `add_`), restated from memory of the un-vendored source, with the
  single-process case of its `all_reduce`.  Its buffers are [dim, n_embed], as there.
"""
from __future__ import annotations

from typing import Tuple

import torch
import torch.nn.functional as F


def rows(z: torch.Tensor) -> torch.Tensor:
    """[B, D, H, W] -> [B*H*W, D] in the quantizer's row order (b, h, w)."""
    return z.permute(0, 2, 3, 1).reshape(-1, z.shape[1])


def ema_update_fp64(flat: torch.Tensor, idx: torch.Tensor, cluster_size: torch.Tensor, embed_avg: torch.Tensor, decay: float,
                    eps: float, count_scale: float = 1.0) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """flat [N, D] rows, idx [N] their codes, cluster_size [K], embed_avg [K, D] (the pre-step state) -> float64
    (cluster_size, embed_avg, codebook) after one update.  `count_scale` multiplies count and S (a stats reducer that
    scales them)."""
    K = cluster_size.shape[0]
    z = flat.to(torch.float64)
    idx = idx.to(torch.int64)
    count = torch.bincount(idx, minlength=K).to(torch.float64) * count_scale
    S = torch.zeros(K, z.shape[1], dtype=torch.float64).index_add_(0, idx, z) * count_scale
    cs = decay * cluster_size.to(torch.float64) + (1 - decay) * count
    ea = decay * embed_avg.to(torch.float64) + (1 - decay) * S
    n = cs.sum()
    smoothed = (cs + eps) / (n + K * eps) * n
    return cs, ea, ea / smoothed[:, None]


def rosinality_train_step(flatten: torch.Tensor, embed_ind: torch.Tensor, embed: torch.Tensor, cluster_size: torch.Tensor,
                          embed_avg: torch.Tensor, decay: float, eps: float) -> None:
    """In place, float32: embed [dim, n_embed], cluster_size [n_embed], embed_avg [dim, n_embed]; flatten [N, dim]."""
    n_embed = embed.shape[1]
    embed_onehot = F.one_hot(embed_ind, n_embed).type(flatten.dtype)
    embed_onehot_sum = embed_onehot.sum(0)
    embed_sum = flatten.transpose(0, 1) @ embed_onehot
    cluster_size.data.mul_(decay).add_(embed_onehot_sum, alpha=1 - decay)
    embed_avg.data.mul_(decay).add_(embed_sum, alpha=1 - decay)
    n = cluster_size.sum()
    cluster_size = (cluster_size + eps) / (n + n_embed * eps) * n
    embed_normalized = embed_avg / cluster_size.unsqueeze(0)
    embed.data.copy_(embed_normalized)
