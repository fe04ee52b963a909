"""CPU checks of tests/oracle_vq_search.py: the decision-rule model is what it claims to be, the grid data make it exact,
the planted structures are what their names say, and every GPU case of tests/test_gpu_vq_search.py lands on the exact-kernel
variant it names with its grid-stride loop turning over.  No GPU needed."""
import numpy as np
import pytest
import torch

import oracle_vq_search as os_
from oracle import vq as ov


@pytest.mark.parametrize("codebook", ["init", "trained"])
def test_rule_matches_the_fp32_oracle_outside_ties(codebook):
    g = torch.Generator().manual_seed(3)
    z = 0.5 * torch.randn(4, 64, 16, 16, generator=g)
    E = (torch.rand(512, 64, generator=g) * 2 - 1) / 512 if codebook == "init" else 0.5 * torch.randn(512, 64, generator=g)
    ties = ov.tie_rows(z, E)
    assert int(ties.sum()) < 0.05 * ties.numel()
    mism = os_.rule_indices(z, E) != ov.code_indices(z, E)
    assert not bool((mism & ~ties).any())


@pytest.mark.parametrize("K,D", [(512, 64), (37, 3), (64, 301)])
def test_rule_matches_integer_brute_force_on_the_coarse_grid(K, D):
    """Coarse grid: every step of the rule is exact, so it is the first minimum of sum (Z - E)^2 in integers -- with
    duplicated codes, exact ties are planted and the first index must win."""
    g = torch.Generator().manual_seed(K + D)
    E = os_.coarse_grid((K, D), g, lim=4)
    E[K - K // 2:] = E[:K // 2].clone()                      # exact duplicates: ties everywhere
    z = os_.coarse_grid((3000, D), g, lim=4)
    Zi, Ei = (z * 16).long(), (E * 16).long()
    d = ((Zi[:, None, :] - Ei[None, :, :]) ** 2).sum(2)
    assert torch.equal(os_.rule_indices(z, E), torch.argmin(d, 1))
    assert int(os_.rule_indices(z, E).max()) < K - K // 2 or K == 1


def test_grid_sums_are_exact_in_float64():
    """The premise of the model: float64 sums of grid data equal the integer sums, up to D = 2048 and rows scaled by
    2^12, so every summation order the kernels use gives the same float64 value."""
    g = torch.Generator().manual_seed(1)
    for D, scale in ((64, 1.0), (64, 2.0 ** 12), (2048, 1.0), (301, 2.0 ** 10)):
        z = os_.fine_grid((200, D), g) * scale
        E = os_.fine_grid((64, D), g)
        Zi, Ei = (z / (os_.FINE * scale)).long(), (E / os_.FINE).long()
        assert int(Zi.abs().max()) <= 4096 and int(Ei.abs().max()) <= 4096
        dot = z.double() @ E.double().t()
        assert torch.equal(dot, (Zi @ Ei.t()).double() * (os_.FINE * os_.FINE * scale))
        assert torch.equal((z.double() ** 2).sum(1), (Zi * Zi).sum(1).double() * (os_.FINE * scale) ** 2)
        perm = torch.randperm(D, generator=g)
        assert torch.equal(z.double()[:, perm] @ E.double()[:, perm].t(), dot)


@pytest.mark.parametrize("name", os_.NON_FINITE)
def test_rule_on_non_finite_inputs_is_torch_argmin(name):
    """On the coarse grid the fp32 oracle's distances are exact too: the model must reproduce torch.argmin over them,
    NaN first, including its NaN and inf rows."""
    z, E = os_.non_finite_case(name)
    dist = ov.distances_fp32(ov.flatten_nchw(z), E)
    want = torch.argmin(dist, 1)
    got = os_.rule_indices(z, E)
    assert torch.equal(got, want)
    nan_rows = torch.isnan(dist).any(1)
    assert bool(nan_rows.any())
    assert torch.equal(got[nan_rows], torch.isnan(dist[nan_rows]).int().argmax(1))       # the first NaN
    if name == "nan_codebook_row":
        assert bool((got == 37).all())
    if name == "nan_and_inf_latents":
        HW, W = 16 * 20, 20
        assert int(got[3 * HW + 4 * W + 4]) == 0 and bool(torch.isinf(dist[3 * HW + 4 * W + 4]).all())


def test_code_positions_follow_the_epilogue_layout():
    for j in range(512):
        gr, ch, k, i3 = os_.position(j)
        assert os_.code_at(gr, ch, k, i3) == j
        c = j % 32
        assert k == ((2 * (c // 4) + (c % 4 >= 2)) & 3)           # epi_chunk: tr[(2q) & 3] / tr[(2q + 1) & 3]


@pytest.mark.parametrize("variant", os_.VARIANTS)
@pytest.mark.parametrize("structure", sorted(os_.tie_structures()))
def test_planted_structures_decide_as_named(structure, variant):
    """The center rows' nearest codes are the planted ones, equidistant or a quantum apart as named, and the tensor
    path's re-check count is predictable (no tile on a binade boundary of its key scale)."""
    codes = os_.tie_structures()[structure]
    assert len(set(codes)) == len(codes)
    z, E = os_.planted_case(structure, variant)
    flat = os_.rows(z)
    got = os_.rule_indices(flat[:1], E)
    want = {"tie": min(codes), "step": codes[0], "step_rev": codes[-1]}[variant]
    assert int(got) == want
    s = os_.exact_scores(flat[:1], E)[0]
    planted = s[codes] - s[codes].min()
    assert planted.max() <= (len(codes) - 1) * os_.QUANTUM and float(s[[j for j in range(512) if j not in codes]].min() - s.min()) > 1.0
    lo, hi = os_.expected_rechecks(flat, E)
    assert lo >= flat.shape[0] // 3                          # every center row: its planted codes are within the threshold
    assert hi < flat.shape[0]


@pytest.mark.parametrize("case", sorted(os_.EXACT_CASES))
def test_exact_cases_land_on_their_variant_and_turn_the_grid(case):
    K, D, (B, H, W), variant = os_.EXACT_CASES[case]
    assert os_.exact_variant(K, D) == variant
    assert os_.exact_passes(B * H * W, K, D) >= 2
    if variant == "staged":
        assert os_.exact_passes(B * H * W, K, D) >= 3 and (B * H * W) % 4 != 0
    assert 10_000 <= B * H * W <= 16_000


def test_exact_kernel_limits():
    warps, smax = os_.exact_kernel_constants()
    assert warps == 8 and smax == 220 * 1024
    assert os_.exact_variant(558, 64) == "staged" and os_.exact_variant(559, 64) == "unstaged"
    assert os_.exact_variant(6200, 64) == "unstaged" and os_.exact_variant(os_.REJECTED_K, 64) == "rejected"
    K, D, (B, H, W), variant = os_.MISALIGNED_CASE
    assert os_.exact_variant(K, D) == variant and os_.exact_passes(B * H * W, K, D) >= 3
    # one pass: 32 rows x 148 CTAs (staged) or 1 row x 8 warps x 592 CTAs (unstaged)
    assert os_.exact_passes(4736, 512, 64) == 1 and os_.exact_passes(4737, 512, 64) == 2
    assert os_.exact_passes(4736, 2048, 64) == 1 and os_.exact_passes(4737, 2048, 64) == 2
    assert np.isclose(os_.recheck_threshold(512.0) / os_.QUANTUM, 2.5)
