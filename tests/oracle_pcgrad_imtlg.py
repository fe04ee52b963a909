"""CPU oracles of the PCGrad and IMTL-G weightings (test infrastructure; the product never imports this module).

Neither weighting is in the reference tree: both live in the un-vendored dependency torchjd (requirements.txt:58, no
commit pin), selectable as `--aggregator pcgrad` / `imtlg` (main.py:1196-1220).  What follows is restated from torchjd's
`PCGradWeighting.forward` and `IMTLGWeighting.forward` as recalled, like the UPGrad oracle (SURVEY App. A) -- parity
unpinned by reference code.  G32 is the float32 Gramian: the arbiter's float64 `J J^T` rounded to float32 once
(oracle.aggregation.arbiter_gramian), which is also what the kernels solve on.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np
import torch

FP32_EPS = float(torch.finfo(torch.float32).eps)


def draw_permutations(k: int) -> list:
    """One PCGrad aggregation's host RNG consumption: k `torch.randperm(k)` calls on the default CPU generator, the
    permutation of chain i drawn i-th."""
    return [torch.randperm(k) for _ in range(k)]


def pcgrad_weights(G32: torch.Tensor, perms: Sequence[torch.Tensor]) -> torch.Tensor:
    """[torchjd-recall] PCGradWeighting.forward, the literal float32 loop: chain i starts at e_i; for j in perms[i], j != i,
    ip = G[j] @ c and, when ip < 0, c[j] -= ip / G[j, j]; w = the chains summed in order i = 0..k-1."""
    G32 = G32.to(torch.float32)
    k = G32.shape[0]
    w = torch.zeros(k, dtype=torch.float32)
    for i in range(k):
        c = torch.zeros(k, dtype=torch.float32)
        c[i] = 1.0
        for j in perms[i].tolist():
            if j == i:
                continue
            ip = G32[j] @ c
            if ip < 0.0:
                c[j] -= ip / G32[j, j]
        w = w + c
    return w


def pcgrad_gradient_space(J: torch.Tensor, perms: Sequence[torch.Tensor]) -> torch.Tensor:
    """Yu et al. 2020 ("Gradient Surgery for Multi-Task Learning", Alg. 1) in P-space, float64: g_i^PC = g_i, then for j in
    perms[i], j != i, g_i^PC -= (g_i^PC . g_j) / |g_j|^2 g_j when g_i^PC . g_j < 0; returns sum_i g_i^PC.  An independent
    cross-check of the Gramian formulation: <g_j, g_i^PC> = (G c)_j when g_i^PC = J^T c."""
    J = J.to(torch.float64)
    out = torch.zeros(J.shape[1], dtype=torch.float64)
    for i in range(J.shape[0]):
        g = J[i].clone()
        for j in perms[i].tolist():
            if j == i:
                continue
            ip = g @ J[j]
            if ip < 0.0:
                g = g - ip / (J[j] @ J[j]) * J[j]
        out += g
    return out


def imtlg_weights(G32: torch.Tensor) -> torch.Tensor:
    """[torchjd-recall] IMTLGWeighting.forward, the literal float32 torch expression."""
    G32 = G32.to(torch.float32)
    d = torch.sqrt(torch.diag(G32))
    v = torch.linalg.pinv(G32) @ d
    s = v.sum()
    return torch.zeros_like(v) if bool(s.abs() < 1e-12) else v / s


def imtlg_weights_fp64(G32: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """The arbiter: the same weights from a float64 eigen-decomposition of the float32-valued Gramian, with pinv's
    tolerance (eigenvalues |l| <= k eps32 max|l| dropped; the singular values of a symmetric matrix are |l|).
    Returns (w float32, number of kept eigenvalues)."""
    G = G32.to(torch.float32).to(torch.float64).numpy()
    k = G.shape[0]
    lam, V = np.linalg.eigh(G)
    tol = k * FP32_EPS * float(np.abs(lam).max())
    keep = np.abs(lam) > tol
    d = torch.sqrt(torch.diag(G32.to(torch.float32))).to(torch.float64).numpy()
    Vk = V[:, keep]
    v = Vk @ ((Vk.T @ d) / lam[keep])
    s = float(v.sum())
    w = np.zeros(k) if abs(s) < 1e-12 else v / s
    return torch.from_numpy(w).to(torch.float32), int(keep.sum())
