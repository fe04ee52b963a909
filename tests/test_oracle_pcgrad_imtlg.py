"""CPU checks of the PCGrad / IMTL-G oracles (tests/oracle_pcgrad_imtlg.py) and of the host side of the two aggregators:
known answers, PCGrad's Gramian loop against the P-space formulation of Yu et al. 2020, IMTL-G's defining property, and
PCGrad's host RNG consumption."""
import numpy as np
import pytest
import torch

import oracle_pcgrad_imtlg as op
from oracle import aggregation as oa

KAT_J = torch.tensor([[-4.0, 1.0, 1.0], [6.0, 1.0, 1.0]])


def random_J(k, P, seed, conflict=True):
    g = torch.Generator().manual_seed(seed)
    J = torch.randn(k, P, generator=g, dtype=torch.float64)
    if conflict:     # pairs of rows pointing against each other: PCGrad has projections to make
        J[1::2] -= 0.8 * J[0:k - 1:2]
    return J.to(torch.float32)


def test_known_answers_torchjd_docstrings():
    G = oa.arbiter_gramian(KAT_J)
    perms = [torch.tensor([0, 1]), torch.tensor([1, 0])]
    w = op.pcgrad_weights(G, perms)
    np.testing.assert_allclose(w.numpy(), [2.2222, 1.5789], atol=5e-5)
    np.testing.assert_allclose((w @ KAT_J).numpy(), [0.5848, 3.8012, 3.8012], atol=5e-5)
    for f in (op.imtlg_weights, lambda G: op.imtlg_weights_fp64(G)[0]):
        w = f(G)
        np.testing.assert_allclose(w.numpy(), [0.5923, 0.4077], atol=5e-5)
        np.testing.assert_allclose((w @ KAT_J).numpy(), [0.0767, 1.0000, 1.0000], atol=5e-5)


@pytest.mark.parametrize("k", [2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("seed", [0, 1])
def test_pcgrad_gramian_loop_equals_gradient_space_projection(k, seed):
    J = random_J(k, 64, 10 * k + seed)
    torch.manual_seed(seed)
    perms = op.draw_permutations(k)
    w = op.pcgrad_weights(oa.arbiter_gramian(J), perms)
    g = op.pcgrad_gradient_space(J, perms)
    np.testing.assert_allclose((w.double() @ J.double()).numpy(), g.numpy(), rtol=1e-4, atol=1e-4 * float(g.abs().max()))
    assert not torch.equal(w, torch.ones(k))           # the conflicting rows were projected


def test_pcgrad_orthogonal_rows_and_zero_row():
    J = torch.zeros(4, 16)
    for i in range(3):
        J[i, 4 * i:4 * i + 4] = torch.arange(1.0, 5.0) * (i + 1)
    perms = [torch.randperm(4) for _ in range(4)]
    np.testing.assert_array_equal(op.pcgrad_weights(oa.arbiter_gramian(J), perms).numpy(), np.ones(4))


@pytest.mark.parametrize("k", [2, 3, 5, 8])
def test_imtlg_defining_property_on_full_rank_jacobians(k):
    J = random_J(k, 200, 7 * k, conflict=False)
    G = oa.arbiter_gramian(J)
    w64, rank = op.imtlg_weights_fp64(G)
    assert rank == k
    for w in (w64, op.imtlg_weights(G)):
        assert abs(float(w.sum()) - 1.0) < 1e-5
        ratio = (G.double() @ w.double()) / torch.sqrt(torch.diag(G).double())   # (G w)_i / |g_i|: equal projections
        np.testing.assert_allclose(ratio.numpy(), float(ratio.mean()), rtol=1e-4)
    np.testing.assert_allclose(op.imtlg_weights(G).numpy(), w64.numpy(), rtol=1e-4, atol=1e-5)


def test_imtlg_rank_deficient_and_zero_gramian():
    J = random_J(3, 50, 3, conflict=False)
    J[2] = J[0]
    w, rank = op.imtlg_weights_fp64(oa.arbiter_gramian(J))
    assert rank == 2 and abs(float(w.sum()) - 1.0) < 1e-5
    w, rank = op.imtlg_weights_fp64(torch.zeros(3, 3))
    assert rank == 0 and torch.equal(w, torch.zeros(3))


@pytest.mark.parametrize("k", [1, 3, 8])
def test_pcgrad_draws_like_torch_randperm_after_manual_seed(k):
    import movae_b200

    wt = movae_b200.PCGrad().weighting
    torch.manual_seed(123)
    got = [wt.draw(k) for _ in range(3)]
    after = torch.rand(1)
    torch.manual_seed(123)
    want = [torch.stack(op.draw_permutations(k)) for _ in range(3)]
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    assert torch.equal(after, torch.rand(1))           # exactly k randperm(k) calls per aggregation, nothing more
    assert torch.equal(wt.last_perms, got[-1])


def test_factory_names_and_reprs():
    import movae_b200

    assert repr(movae_b200.make_aggregator("pcgrad")) == "PCGrad()"
    assert repr(movae_b200.make_aggregator("IMTLG")) == "IMTLG()"
    assert isinstance(movae_b200.make_aggregator("imtlg").weighting, movae_b200.IMTLGWeighting)
    for name in ("cagrad", "nashmtl"):
        with pytest.raises(ValueError, match="not supported"):
            movae_b200.make_aggregator(name)
