"""CPU tests: the VQ oracle restatement against golden outputs of the reference module
(models/vq_vae.py:11-124 run behind the shim by tests/golden/make_golden.py)."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import vq as ov

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden import load_vq_golden  # noqa: E402

GOLD = load_vq_golden()
TAGS = ("init", "trained", "dup")


@pytest.mark.parametrize("tag", TAGS)
def test_forward_matches_reference_module(tag):
    z = torch.from_numpy(GOLD[f"{tag}_z"])
    E = torch.from_numpy(GOLD[f"{tag}_E"])
    q, commit, embed, idx = ov.quantize_forward(z, E)
    ties = ov.tie_rows(z, E)
    mism = idx.numpy() != GOLD[f"{tag}_idx"]
    # same ops, same library -> identical except (possibly) on fp32-tie rows if the BLAS differs
    assert not np.any(mism & ~ties.numpy()), f"{mism.sum()} mismatches outside tie rows"
    if not mism.any():
        np.testing.assert_array_equal(q.numpy(), GOLD[f"{tag}_q"])
    assert float(commit) == pytest.approx(float(GOLD[f"{tag}_commit"]), rel=1e-6)
    assert float(embed) == pytest.approx(float(GOLD[f"{tag}_embed"]), rel=1e-6)
    assert ov.codebook_usage_percentage(idx, E.shape[0]) == pytest.approx(float(GOLD[f"{tag}_usage"]))


def test_duplicate_codebook_rows_pick_first_index():
    idx = GOLD["dup_idx"]
    assert idx.max() < 256   # rows 256.. duplicate 0..255; torch.argmin returns the first minimum


@pytest.mark.parametrize("tag", TAGS)
def test_closed_form_backward_matches_reference_autograd(tag):
    z = torch.from_numpy(GOLD[f"{tag}_z"])
    E = torch.from_numpy(GOLD[f"{tag}_E"])
    idx = torch.from_numpy(GOLD[f"{tag}_idx"])
    dz, dE = ov.quantize_backward(z, E, idx, torch.from_numpy(GOLD[f"{tag}_r"]), 0.7, 1.3)
    np.testing.assert_allclose(dz.numpy(), GOLD[f"{tag}_dz"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(dE.numpy(), GOLD[f"{tag}_dE"], rtol=1e-4, atol=1e-8)


def test_autograd_of_restatement_matches_reference():
    z = torch.from_numpy(GOLD["trained_z"]).requires_grad_(True)
    E = torch.from_numpy(GOLD["trained_E"]).requires_grad_(True)
    q, commit, embed, _ = ov.quantize_forward(z, E)
    (torch.sum(q * torch.from_numpy(GOLD["trained_r"])) + 0.7 * commit + 1.3 * embed).backward()
    np.testing.assert_allclose(z.grad.numpy(), GOLD["trained_dz"], rtol=1e-6, atol=1e-8)
    np.testing.assert_allclose(E.grad.numpy(), GOLD["trained_dE"], rtol=1e-5, atol=1e-9)
