"""CPU checks of VectorQuantizerEMA: its two oracles (tests/oracle_vq_ema.py) agree, the update is one k-means step at
decay 0, the total cluster size follows its recurrence, and the module's host-side contract (validation, state-dict
keys, no gradient on the codebook, CUDA only)."""
import numpy as np
import pytest
import torch

import oracle_vq_ema as oe


def _batch(N, K, D, seed, used=None):
    g = torch.Generator().manual_seed(seed)
    flat = 0.5 * torch.randn(N, D, generator=g)
    idx = torch.randint(0, used or K, (N,), generator=g)
    return flat, idx


@pytest.mark.parametrize("K,D,N,used", [(512, 64, 4096, None), (100, 48, 300, 40), (16, 3, 64, None)])
def test_restatements_agree_over_steps(K, D, N, used):
    decay, eps = 0.9, 1e-5
    E0 = (torch.rand(K, D, generator=torch.Generator().manual_seed(1)) * 2 - 1) / K
    cs, ea = torch.zeros(K, dtype=torch.float64), E0.to(torch.float64)
    embed, cs32, ea32 = E0.t().contiguous(), torch.zeros(K), E0.t().contiguous()
    for step in range(4):
        flat, idx = _batch(N, K, D, 10 + step, used)
        cs, ea, E = oe.ema_update_fp64(flat, idx, cs, ea, decay, eps)
        oe.rosinality_train_step(flat, idx, embed, cs32, ea32, decay, eps)
        np.testing.assert_allclose(cs32.numpy(), cs.numpy(), rtol=1e-6)
        # float32 sums of rows of magnitude ~1, rounded again by mul_ / add_: absolute error ~1e-8 where S cancels
        np.testing.assert_allclose(ea32.t().numpy(), ea.numpy(), rtol=1e-4, atol=1e-7)
        np.testing.assert_allclose(embed.t().numpy(), E.numpy(), rtol=1e-4, atol=1e-7)
        assert np.isfinite(embed.numpy()).all()


def test_decay_zero_is_one_k_means_step():
    K, D, N = 32, 8, 2000
    flat, idx = _batch(N, K, D, 3, used=24)
    cs, ea, E = oe.ema_update_fp64(flat, idx, torch.rand(K), torch.randn(K, D), 0.0, 1e-12)
    for j in range(24):
        np.testing.assert_allclose(E[j].numpy(), flat[idx == j].to(torch.float64).mean(0).numpy(), rtol=1e-9, atol=1e-12)
    np.testing.assert_array_equal(cs.numpy(), torch.bincount(idx, minlength=K).numpy())


def test_total_cluster_size_recurrence():
    K, D, decay = 64, 4, 0.95
    cs, ea = torch.zeros(K, dtype=torch.float64), torch.zeros(K, D, dtype=torch.float64)
    total = 0.0
    for step, N in enumerate((100, 37, 512, 1)):
        flat, idx = _batch(N, K, D, step)
        cs, ea, _ = oe.ema_update_fp64(flat, idx, cs, ea, decay, 1e-5)
        total = decay * total + (1 - decay) * N
        np.testing.assert_allclose(float(cs.sum()), total, rtol=1e-12)


def test_constructor_state_dict_and_gradients():
    import movae_b200

    for bad in (dict(decay=1.0), dict(decay=-0.1), dict(decay=float("nan")), dict(epsilon=0.0), dict(epsilon=-1e-5)):
        with pytest.raises(ValueError):
            movae_b200.VectorQuantizerEMA(512, 64, **bad)
    vq = movae_b200.VectorQuantizerEMA(100, 48, decay=0.8, epsilon=1e-3)
    assert vq.decay == 0.8 and vq.epsilon == 1e-3 and vq.K == 100 and vq.D == 48
    assert set(vq.state_dict()) == {"embedding.weight", "cluster_size", "embed_avg"}
    assert not vq.embedding.weight.requires_grad
    w = vq.embedding.weight.detach()
    assert float(w.abs().max()) <= 1 / 100
    torch.testing.assert_close(vq.embed_avg, w, rtol=0, atol=0)
    assert vq.embed_avg.data_ptr() != w.data_ptr()
    assert torch.count_nonzero(vq.cluster_size) == 0
    assert vq.stats_reducer is None
    assert isinstance(vq, movae_b200.VectorQuantizer)
    other = movae_b200.VectorQuantizerEMA(100, 48)
    other.load_state_dict(vq.state_dict())
    torch.testing.assert_close(other.embedding.weight, vq.embedding.weight, rtol=0, atol=0)


def test_cpu_inputs_raise_cuda():
    import movae_b200

    vq = movae_b200.VectorQuantizerEMA(512, 64)
    with pytest.raises(RuntimeError, match="CUDA"):
        vq(torch.randn(2, 64, 4, 4))
    with pytest.raises(RuntimeError, match="CUDA"):
        vq.eval()(torch.randn(2, 64, 4, 4))
    with pytest.raises(RuntimeError, match="CUDA"):
        vq.get_code_indices(torch.randn(2, 64, 4, 4))
    with pytest.raises(TypeError):
        movae_b200.parallel.install_codebook_allreduce(movae_b200.VectorQuantizer(512, 64))
    movae_b200.parallel.install_codebook_allreduce(vq)
    assert callable(vq.stats_reducer)


def test_c_abi_validates_before_touching_the_device():
    import movae_b200

    lib = movae_b200.lib()
    assert lib.movae_vq_ema_workspace_bytes(-1, 512, 64) == 0
    assert lib.movae_vq_ema_workspace_bytes(0, 512, 64) >= 256 + (512 + 512 * 64) * 4
    assert lib.movae_vq_ema_workspace_bytes(1 << 20, 512, 64) > lib.movae_vq_ema_workspace_bytes(0, 512, 64)
    assert lib.movae_vq_ema_workspace_bytes(1 << 20, 100, 48) == lib.movae_vq_ema_workspace_bytes(0, 100, 48)
    fake = 1 << 20                                                # never dereferenced: validation fails first
    for decay, eps in ((1.0, 1e-5), (-0.5, 1e-5), (0.99, 0.0)):
        assert lib.movae_vq_ema_apply_f32(fake, 512, 64, decay, eps, fake, fake + 4096, fake + 8192, fake + 12288, fake, 1 << 30, None) == 1
        assert "must" in lib.movae_last_error().decode()
