"""TEST INFRASTRUCTURE ONLY: an exact model of the decision rule both codebook searches implement (K4 `vq_argmin_tc.cu`
with its in-kernel re-check, K4x `vq_argmin_exact.cu`), plus data generators on which that model is bit-exact.

The rule, as the kernels document it:
    z^2, e_j^2 and z.e_j are summed in float64 and rounded to float32 once;
    dist_j = fl(fl(z^2 + e_j^2) - 2 z.e_j)   (float32 add, multiply, subtract in that order);
    idx = torch.argmin(dist): the first NaN if there is one, else the first minimum (0 when every distance is inf).

`rule_indices` evaluates exactly that.  It equals the kernels bit for bit whenever their float64 sums are exact, which
is what the grid generators below guarantee: values m 2^-12 with |m| <= 2^12 (optionally times a power of two per row or
per code) have products m m' 2^-24 with |m m'| <= 2^24, and up to 2^11 such terms sum to below 2^35 -- exact in float64
in any order.  The float32 roundings of the sums and of the distance are still real roundings.  On the coarse grid
(m / 16, |m| <= 32) every step is exact, also the tensor path's bf16 split and its float32 accumulation, so planted ties
are exact ties and the tensor path's keys equal the exact scores.
"""
from __future__ import annotations

import math
import os
import re

import numpy as np
import torch

FINE = 2.0 ** -12          # fine grid quantum; |m| <= 2^12
COARSE = 1.0 / 16.0        # coarse grid quantum; |m| <= 32
QUANTUM = COARSE * COARSE  # quantum of squared distances and scores on the coarse grid


def rows(z: torch.Tensor) -> torch.Tensor:
    """[B, D, H, W] -> [N, D] in the search's row order (b, h, w); [N, D] passes through."""
    return z if z.dim() == 2 else z.permute(0, 2, 3, 1).reshape(-1, z.shape[1])


def rule_distances(flat: torch.Tensor, E: torch.Tensor) -> torch.Tensor:
    """float32 [n, K] distances of the rule for rows `flat` [n, D] (CPU, float64 sums rounded once)."""
    f = flat.detach().cpu().double()
    E64 = E.detach().cpu().double()
    z2 = (f * f).sum(1).float()
    e2 = (E64 * E64).sum(1).float()
    dot = (f @ E64.t()).float()
    return (z2[:, None] + e2[None, :]) - 2 * dot


def rule_indices(z: torch.Tensor, E: torch.Tensor, chunk: int = 1 << 15) -> torch.Tensor:
    """int64 [N] (CPU): the index the rule selects for every row of z ([B, D, H, W] or [N, D])."""
    flat = rows(z)
    return torch.cat([torch.argmin(rule_distances(flat[r0:r0 + chunk], E), 1) for r0 in range(0, flat.shape[0], chunk)])


def exact_scores(flat: torch.Tensor, E: torch.Tensor) -> torch.Tensor:
    """float64 [n, K] scores |e_j|^2 - 2 z.e_j (what the tensor path's keys encode); exact on grid data."""
    f = flat.detach().cpu().double()
    E64 = E.detach().cpu().double()
    return (E64 * E64).sum(1)[None, :] - 2.0 * f @ E64.t()


# ---------------------------------------------------------------------------------------------- grid data
def fine_grid(shape, g: torch.Generator, sigma: float = 0.5, device="cpu") -> torch.Tensor:
    """Gaussian-looking float32 values quantized onto m 2^-12, |m| <= 2^12."""
    x = torch.randn(shape, generator=g, device=device) * (sigma / FINE)
    return x.round_().clamp_(-4096, 4096).mul_(FINE)


def coarse_grid(shape, g: torch.Generator, lim: int = 32, device="cpu") -> torch.Tensor:
    """float32 values m / 16, integer |m| <= lim."""
    return torch.randint(-lim, lim + 1, shape, generator=g, device=device, dtype=torch.float32).div_(16.0)


def to_nchw(flat: torch.Tensor, B: int, H: int, W: int) -> torch.Tensor:
    return flat.reshape(B, H, W, -1).permute(0, 3, 1, 2).contiguous()


# ---------------------------------------------------------------------------------------------- tensor-path layout
# Within a 32-code chunk of an epilogue group, code j (from `code_of` in vq_argmin_tc.cu): bits 1-2 name the tracker,
# bit 0 and bits 3-4 are the key's three low mantissa bits (i3); chunk = (j mod 256) / 32, group = j / 256.
def code_at(group: int, chunk: int, tracker: int, i3: int = 0) -> int:
    assert 0 <= group < 2 and 0 <= chunk < 8 and 0 <= tracker < 4 and 0 <= i3 < 8
    return group * 256 + chunk * 32 + ((i3 >> 1) << 3) + (tracker << 1) + (i3 & 1)


def position(j: int):
    """(group, chunk, tracker, i3) of code j."""
    c = j % 32
    return j // 256, (j % 256) // 32, (c >> 1) & 3, (c & 1) | ((c >> 3) << 1)


def plant(E: torch.Tensor, center: torch.Tensor, codes, extra_quanta, radius: int = 16):
    """Codebook rows E[codes[i]] := center + a displacement whose squared length is (radius / 16)^2 + extra_quanta[i]
    QUANTUM, exactly (coarse grid): one channel moved by radius / 16 and, per extra quantum, one more channel by 1 / 16.
    `center` must leave room (|m| <= 32 - radius - 1).  Returns the planted squared distances."""
    D = E.shape[1]
    d2 = []
    for i, (j, q) in enumerate(zip(codes, extra_quanta)):
        v = torch.zeros(D)
        ch = (7 * i) % D
        v[ch] = (radius if i % 2 == 0 else -radius) * COARSE
        for k in range(q):
            v[(ch + 1 + k) % D] = COARSE if k % 2 == 0 else -COARSE
        E[j] = center + v
        d2.append(float((v.double() ** 2).sum()))
    return d2


# ---------------------------------------------------------------------------------------------- tensor-path threshold
def tile_key_scale(z2max: float, emax2_f32: float) -> float:
    """M of a tile, as the producer warps form it (vq_argmin_tc.cu, the tile's key constants), from the tile's max |z|^2
    and the float32 max |e|^2; float32 arithmetic in the kernel's order.  Returns (M, ambiguous): ambiguous when Rg is
    so close to a power of two that a one-ulp difference in the chain could change M."""
    f = np.float32
    emax2 = f(emax2_f32) * f(1.000001)
    emax = f(np.sqrt(emax2)) * f(1.000001)
    craw = f(f(f(2.001) * f(np.sqrt(f(z2max) * f(1.00001)))) * emax) + f(1e-30)
    cb = (int(np.array(craw, dtype=np.float32).view(np.uint32)) + 0xFFFF) >> 16
    C = np.array(cb << 16, dtype=np.uint32).view(np.float32)[()]
    rg = f(max(f(f(2.0) * C + max(emax2, f(f(f(z2max) + emax2) * f(0.03125)))), f(1e-30)) * f(1.001))
    mexp = max((int(np.array(rg, dtype=np.float32).view(np.uint32)) >> 23) + 1, 40)
    M = 2.0 ** (mexp - 127)
    frac = float(rg) / 2.0 ** math.floor(math.log2(float(rg)))
    return M, mexp > 40 and (frac > 2.0 - 1e-5 or frac < 1.0 + 1e-5)


def recheck_threshold(M: float) -> float:
    """Gap below which the epilogue cannot decide a row: 1.25 M 2^-16 (keys live in [M, 2M))."""
    return 1.25 * M * 2.0 ** -16


def expected_rechecks(flat: torch.Tensor, E: torch.Tensor, tile: int = 128):
    """(fewest, most) rows the tensor path must send to its re-check on coarse-grid data, where its keys are the exact
    scores: a row is re-checked iff a second code's score lies within the tile's threshold of the row's best score.
    Rows whose gap is within 8 key quanta of the threshold may go either way."""
    s = exact_scores(flat, E)
    top2 = torch.topk(s, 2, dim=1, largest=False).values
    gap = top2[:, 1] - top2[:, 0]
    z2 = (flat.double() ** 2).sum(1)
    emax2 = float((E.double() ** 2).sum(1).max())
    lo = hi = 0
    for t0 in range(0, flat.shape[0], tile):
        M, amb = tile_key_scale(float(z2[t0:t0 + tile].max()), emax2)
        assert not amb, "tile key scale on a binade boundary: pick other data"
        thr, q8 = recheck_threshold(M), 8 * M * 2.0 ** -23
        g = gap[t0:t0 + tile]
        lo += int((g <= thr - q8).sum())
        hi += int((g <= thr + q8).sum())
    return lo, hi


# ---------------------------------------------------------------------------------------------- exact-kernel launch rules
SMS = 148                       # B200
_SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "mo-vae_b200", "csrc", "vq_argmin_exact.cu")


def exact_kernel_constants():
    """(kExWarps, kExMaxSmem in bytes) parsed from vq_argmin_exact.cu."""
    src = open(_SRC).read()
    warps = int(re.search(r"constexpr int kExWarps = (\d+);", src).group(1))
    m = re.search(r"constexpr size_t kExMaxSmem = (\d+)\s*\*\s*(\d+);", src)
    return warps, int(m.group(1)) * int(m.group(2))


def exact_variant(K: int, D: int) -> str:
    """'staged' (codebook transposed in shared memory, 4 rows per warp), 'unstaged' (1 row per warp, codebook from
    global memory) or 'rejected' -- launch_vq_argmin_exact's choice."""
    warps, smax = exact_kernel_constants()
    staged = (warps * 4 * (D + K) + K + D * (K + 1)) * 4
    plain = (warps * 1 * (D + K) + K) * 4
    return "staged" if staged <= smax else ("unstaged" if plain <= smax else "rejected")


def exact_passes(N: int, K: int, D: int, sms: int = SMS) -> int:
    """Grid-stride passes the busiest warp of the exact kernel makes over N rows."""
    warps, _ = exact_kernel_constants()
    v = exact_variant(K, D)
    R = 4 if v == "staged" else 1
    groups = -(-N // R)
    grid = max(1, min(-(-groups // warps), sms if v == "staged" else 4 * sms))
    return -(-groups // (grid * warps))


# ---------------------------------------------------------------------------------------------- cases
# exact kernel: name -> (K, D, (B, H, W), variant it must land on); N mod 4 != 0 where staged (the last group of 4 rows
# repeats its final row), at least two grid-stride passes everywhere
EXACT_CASES = {
    "staged_K512": (512, 64, (3, 61, 83), "staged"),
    "staged_K558": (558, 64, (3, 61, 83), "staged"),
    "unstaged_K559": (559, 64, (2, 73, 79), "unstaged"),
    "unstaged_K2048": (2048, 64, (2, 73, 79), "unstaged"),
    "unstaged_K6200": (6200, 64, (2, 73, 79), "unstaged"),
    "K1": (1, 64, (2, 61, 83), "staged"),
    "K2": (2, 64, (2, 61, 83), "staged"),
    "K31": (31, 64, (2, 61, 83), "staged"),
    "K100": (100, 64, (2, 61, 83), "staged"),
    "D3": (512, 3, (2, 61, 83), "staged"),
    "D300": (100, 300, (2, 61, 83), "staged"),
    "D301_scalar_staging": (100, 301, (2, 61, 83), "staged"),
    "D2048_unstaged": (64, 2048, (2, 61, 83), "unstaged"),
}
MISALIGNED_CASE = (512, 64, (3, 61, 83), "staged")       # codebook view one float past a 16-byte boundary
REJECTED_K = 6201                                          # at D = 64: the first codebook neither variant can hold


def tie_structures():
    """name -> codes planted equidistant (or a quantum apart) around one row, at chosen tracker / chunk / group positions
    of the tensor path (K = 512)."""
    S = {}
    for n in (2, 3, 4, 5):
        S[f"one_tracker_across_chunks_{n}"] = [code_at(0, c, 1, c % 8) for c in (1, 3, 4, 6, 7)[:n]]
        S[f"trackers_of_one_group_{n}"] = [code_at(1, 2 + i // 4, i % 4, 5) for i in range(n)]
        S[f"across_groups_{n}"] = [code_at(i % 2, 3 + i // 2, (i + 1) % 4, 2) for i in range(n)]
        S[f"one_tracker_one_chunk_{n}"] = [code_at(0, 4, 3, i3) for i3 in (6, 1, 3, 0, 7)[:n]]
    S["one_per_tracker_both_groups"] = [code_at(g, 5, k, 3) for g in (0, 1) for k in range(4)]
    S["winner_after_first_tracker"] = [code_at(0, 0, 3, 0), code_at(0, 1, 0, 0)]          # k1 = tracker 0, winner tracker 3
    S["winner_has_larger_key_bits"] = [code_at(0, 1, 2, 7), code_at(0, 5, 2, 0)]          # same tracker: smaller key, later index
    # three trackers of one group within the threshold: the exchange carries two codes, the tied winner (largest key bits,
    # lowest index) is the third -- only the n_close > 1 scan finds it
    S["winner_is_third_close_tracker"] = [code_at(0, 0, 2, 7), code_at(0, 1, 0, 0), code_at(0, 1, 1, 0)]
    return S


VARIANTS = ("tie", "step", "step_rev")          # all equidistant; code i one quantum farther than i - 1; the reverse


def planted_case(structure: str, variant: str, B: int = 2, H: int = 148, W: int = 128, seed: int = 0):
    """(z [B, 64, H, W], E [512, 64]) on the coarse grid: a random codebook with the structure planted around one
    center; every third row is the center, the others are random rows."""
    g = torch.Generator().manual_seed(seed + 101 * sorted(tie_structures()).index(structure) + VARIANTS.index(variant))
    codes = tie_structures()[structure]
    E = coarse_grid((512, 64), g)
    center = coarse_grid((64,), g, lim=10)
    n = len(codes)
    quanta = {"tie": [0] * n, "step": list(range(n)), "step_rev": list(range(n))[::-1]}[variant]
    plant(E, center, codes, quanta)
    flat = coarse_grid((B * H * W + 77, 64), g)[:B * H * W]
    flat[::3] = center
    return to_nchw(flat, B, H, W), E


def non_finite_case(name: str, seed: int = 0):
    """(z [4, 64, 16, 20], E [512, 64]) on the coarse grid with the named non-finite entries."""
    g = torch.Generator().manual_seed(seed)
    z = coarse_grid((4, 64, 16, 20), g)
    E = coarse_grid((512, 64), g)
    if name == "nan_codebook_row":
        E[37, 5] = float("nan")
    elif name == "inf_codebook_entry":
        E[300, 11] = float("inf")
    elif name == "nan_and_inf_latents":
        z[0, 3, 0, 1] = float("nan")
        z[1, 7, 2, 3] = float("inf")
        z[2, 9, 5, 5] = float("-inf")
        z[0, :, 0, 0] = float("inf")
        z[3, :, 4, 4] = 1e20                      # |z|^2 overflows float32: every distance is inf
        z[2, 5, 1, 1] = -3e19
    else:
        raise ValueError(name)
    return z, E


NON_FINITE = ("nan_codebook_row", "inf_codebook_entry", "nan_and_inf_latents")
