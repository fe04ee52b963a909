"""GPU tests of the L2 hand-off inside the fused aggregation launch (csrc/aggregate.cu): each pass loads a CTA's steps
with an L2 eviction priority that depends on the step's distance from the back of the deal.  The fused gradient is
compared bit for bit with K3 (`ops.recombine`, which loads every tile alike) applied to the weights the launch returned,
at sizes where J is far larger than the L2, so that steps inside and outside the L2 window both occur."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def synthetic_J(k, P, seed, ld=None):
    ld = P if ld is None else ld
    g = torch.Generator(device="cuda").manual_seed(seed)
    base = torch.randn(k, ld, generator=g, device="cuda") * torch.logspace(0, -1, k, device="cuda")[:, None]
    return base[:, :P]


@pytest.fixture(scope="module")
def mv():
    import movae_b200
    return movae_b200


def fused(mv, J, out=None, accumulate=False, want_grad=True):
    spec, vec, aux = mv.make_aggregator("upgrad").weighting.solve_spec(J.shape[0])
    return mv.ops.aggregate(J, spec, vec, aux, out=out, accumulate=accumulate, want_grad=want_grad)


def round_items():
    """float4 items in one round of whole k = 3 tiles (256 threads x 4 float4 per CTA, two CTAs per SM)."""
    return 1024 * 2 * torch.cuda.get_device_properties(0).multi_processor_count


def check_against_k3(mv, J, out=None, accumulate=False):
    before = None if out is None else out.clone()
    w, diag, G, g = fused(mv, J, out=out, accumulate=accumulate)
    ref = mv.ops.recombine(J, w, out=before, accumulate=accumulate)
    torch.cuda.synchronize()
    assert torch.isfinite(w).all()
    assert torch.equal(g, ref)
    return w, G, g


@pytest.mark.parametrize("shape", ["remainder", "whole_rounds", "ragged"])
def test_k3_large_matches_k3_recombine(mv, shape):
    # 480 MB at k = 3: steps outside and inside the L2 window; with a remainder slice, without one, with a ragged tail
    P = {"remainder": 40_000_000, "whole_rounds": 4 * 33 * round_items(), "ragged": 40_000_003}[shape]
    check_against_k3(mv, synthetic_J(3, P, P % 97))


def test_ld_larger_than_P(mv):
    P = 40_000_003
    check_against_k3(mv, synthetic_J(3, P, 5, ld=P + 9))           # ldJ % 4 == 0: float4 path with a ragged tail
    check_against_k3(mv, synthetic_J(3, P, 6, ld=P + 5))           # ldJ % 4 != 0: scalar path


@pytest.mark.parametrize("shape", ["one_tile_per_cta", "partial_grid", "one_round_and_remainder"])
def test_deals_inside_the_window(mv, shape):
    # a CTA has one tile, or one tile and a remainder slice: every step is inside the L2 window
    P = {"one_tile_per_cta": 4 * 1024 * 100, "partial_grid": 1_000_000,
         "one_round_and_remainder": 4 * round_items() + 4 * 5000 + 3}[shape]
    check_against_k3(mv, synthetic_J(3, P, 11))


def test_accumulate(mv):
    P = 40_000_000
    J = synthetic_J(3, P, 21)
    out = torch.randn(P, generator=torch.Generator(device="cuda").manual_seed(22), device="cuda")
    check_against_k3(mv, J, out=out, accumulate=True)


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6, 7, 8])
def test_every_k_at_large_P(mv, k):
    check_against_k3(mv, synthetic_J(k, 30_000_001, 40 + k))


def test_weights_only_then_full_launch(mv):
    J = synthetic_J(3, 40_000_000, 31)
    w0, _, G0, _ = fused(mv, J, want_grad=False)
    w1, G1, _ = check_against_k3(mv, J)
    assert torch.equal(w0, w1) and torch.equal(G0, G1)


def test_repeated_launches_are_bit_identical(mv):
    J = synthetic_J(3, 40_000_000, 32)
    runs = [fused(mv, J) for _ in range(3)]
    torch.cuda.synchronize()
    for w, diag, G, g in runs[1:]:
        assert torch.equal(w, runs[0][0]) and torch.equal(diag, runs[0][1])
        assert torch.equal(G, runs[0][2]) and torch.equal(g, runs[0][3])
