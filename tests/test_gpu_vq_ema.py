"""GPU tests of VectorQuantizerEMA: the search, gather, losses and latent gradients equal VectorQuantizer's from the same
pre-step codebook, and the codebook update equals the float64 oracle (tests/oracle_vq_ema.py) started from the module's
own pre-step state.

Bars: indices, quantized, losses and dz bit-exact against VectorQuantizer (the same kernels); cluster_size rtol 1e-6;
embed_avg rtol 1e-4 / atol 1e-8 (float32 sums of up to N rows, the bar of the codebook gradient) and the codebook with
that absolute bar carried through the division by smoothed_j.  K = 512, D = 64 is bit-reproducible run to run; other
shapes sum with float32 atomics and are checked to tolerance only."""
import os
import socket

import numpy as np
import pytest
import torch

import oracle_vq_ema as oe

pytestmark = pytest.mark.gpu

DECAY, EPS = 0.99, 1e-5


@pytest.fixture(scope="module")
def mv():
    import movae_b200
    return movae_b200


@pytest.fixture(scope="module")
def ov():
    from oracle import vq
    return vq


def make_z(B, D, H, W, seed):
    return 0.5 * torch.randn(B, D, H, W, generator=torch.Generator().manual_seed(seed))


def trained_codebook(K, D, seed):
    return 0.5 * torch.randn(K, D, generator=torch.Generator().manual_seed(seed))


def pair(mv, E, trained_state=False, **kw):
    """(VectorQuantizerEMA, VectorQuantizer) on cuda with codebook E.  trained_state: cluster_size ~ 20 per code and
    embed_avg = E * cluster_size, the state of a codebook that has been following its averages for a while."""
    K, D = E.shape
    ema = mv.VectorQuantizerEMA(K, D, **kw).cuda()
    ref = mv.VectorQuantizer(K, D).cuda()
    with torch.no_grad():
        ema.embedding.weight.copy_(E)
        ref.embedding.weight.copy_(E)
        if trained_state:
            cs = 15.0 + 10.0 * torch.rand(K, generator=torch.Generator().manual_seed(K))
            ema.cluster_size.copy_(cs)
            ema.embed_avg.copy_(E * cs[:, None])
        else:
            ema.embed_avg.copy_(E)
    return ema, ref


def state(vq):
    return {n: t.detach().cpu().clone() for n, t in (("E", vq.embedding.weight), ("cs", vq.cluster_size), ("ea", vq.embed_avg))}


def check_update(vq, pre, z, idx, count_scale=1.0):
    """The module's state after one training forward == the float64 oracle from its own pre-step state `pre`."""
    cs, ea, E = oe.ema_update_fp64(oe.rows(z), idx.cpu(), pre["cs"], pre["ea"], vq.decay, vq.epsilon, count_scale)
    post = state(vq)
    np.testing.assert_allclose(post["cs"].numpy(), cs.numpy(), rtol=1e-6)
    np.testing.assert_allclose(post["ea"].numpy(), ea.numpy(), rtol=1e-4, atol=1e-8)
    n = cs.sum()
    smoothed = ((cs + vq.epsilon) / (n + cs.numel() * vq.epsilon) * n).numpy()
    got, want, atol = post["E"].numpy(), E.numpy(), (1e-8 / smoothed)[:, None]
    err = np.abs(got - want) - (atol + 1e-4 * np.abs(want))
    assert (err <= 0).all(), f"codebook: {int((err > 0).sum())} elements off, worst excess {err.max():.3g}"
    assert np.isfinite(post["E"].numpy()).all()


def one_step_parity(mv, ema, ref, z, seed=1):
    """One training forward + backward of both classes from the same codebook: everything VectorQuantizer computes for
    the latents is bit-identical; the update equals the oracle."""
    pre = state(ema)
    r = torch.randn(z.shape, generator=torch.Generator().manual_seed(seed)).cuda()
    outs = []
    for vq in (ema, ref):
        zc = z.cuda().requires_grad_(True)
        q, commit, embed, idx = vq(zc)
        (torch.sum(q * r) + 0.7 * commit + 1.3 * embed).backward()
        outs.append((q.detach().cpu(), float(commit), float(embed), idx.cpu(), zc.grad.cpu()))
    (q, c, e, idx, dz), (q_r, c_r, e_r, idx_r, dz_r) = outs
    assert torch.equal(idx, idx_r)
    assert torch.equal(q, q_r)
    assert c == c_r and e == e_r
    assert torch.equal(dz, dz_r)
    assert ema.embedding.weight.grad is None
    check_update(ema, pre, z, idx)
    return idx


# ----------------------------------------------------------------------------------------------- one-step parity
@pytest.mark.parametrize("shape", [(16, 8, 8), (4, 32, 32), (2, 64, 64), (1, 4, 8)], ids=["hw64", "hw1024", "hw4096_N8192", "N32"])
@pytest.mark.parametrize("trained", [False, True], ids=["fresh", "trained_state"])
def test_one_step_k512_tma_path(mv, shape, trained):
    B, H, W = shape
    ema, ref = pair(mv, trained_codebook(512, 64, 1), trained_state=trained)
    one_step_parity(mv, ema, ref, make_z(B, 64, H, W, B * H))


@pytest.mark.parametrize("shape", [(3, 7, 9), (7, 4, 5), (40, 5, 13), (1, 1, 100), (2, 3, 5)],
                         ids=["ragged_hw63", "hw20", "hw65_N2600", "N100", "N30"])
def test_one_step_k512_ragged_and_small(mv, shape):
    B, H, W = shape
    ema, ref = pair(mv, trained_codebook(512, 64, 2), trained_state=True)
    one_step_parity(mv, ema, ref, make_z(B, 64, H, W, B + H * W))


@pytest.mark.parametrize("K,D,shape", [(100, 48, (3, 5, 7)), (512, 32, (4, 8, 8)), (1024, 64, (2, 8, 8)), (256, 64, (4, 8, 8))])
def test_one_step_other_shapes(mv, K, D, shape):
    B, H, W = shape
    ema, ref = pair(mv, trained_codebook(K, D, K + D), trained_state=True)
    one_step_parity(mv, ema, ref, make_z(B, D, H, W, K + D))


# ----------------------------------------------------------------------------------------------- trajectories
@pytest.mark.parametrize("K,D,shape", [(512, 64, (8, 16, 16)), (512, 64, (5, 7, 9)), (100, 48, (4, 8, 8))])
def test_five_step_trajectory(mv, ov, K, D, shape):
    """Each step from the module's own state; and, on a trained-like codebook without tie rows, the whole trajectory
    against the oracle run on its own (its own search with its own float32-rounded codebook)."""
    B, H, W = shape
    E0 = trained_codebook(K, D, 7)
    ema, _ = pair(mv, E0, trained_state=True)
    cs_o, ea_o = ema.cluster_size.cpu().double(), ema.embed_avg.cpu().double()
    E_o = E0.clone()
    for step in range(5):
        z = make_z(B, D, H, W, 100 + step)
        pre = state(ema)
        _, _, _, idx = ema(z.cuda())
        check_update(ema, pre, z, idx)
        assert not ov.tie_rows(z, E_o).any()
        idx_o = ov.code_indices(z, E_o)
        assert torch.equal(idx.cpu(), idx_o), f"step {step}: the module's search left the oracle's trajectory"
        cs_o, ea_o, E64 = oe.ema_update_fp64(oe.rows(z), idx_o, cs_o, ea_o, DECAY, EPS)
        E_o = E64.to(torch.float32)
    np.testing.assert_allclose(ema.cluster_size.cpu().numpy(), cs_o.numpy(), rtol=1e-6)
    np.testing.assert_allclose(ema.embed_avg.cpu().numpy(), ea_o.numpy(), rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(ema.embedding.weight.cpu().numpy(), E_o.numpy(), rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("shape", [(16, 32, 32), (7, 15, 15)], ids=["tma", "cp_async"])
def test_k512_update_is_bit_reproducible(mv, shape):
    B, H, W = shape
    E = trained_codebook(512, 64, 3)
    z = make_z(B, 64, H, W, 5).cuda()
    results = []
    for _ in range(2):
        ema, _ = pair(mv, E, trained_state=True)
        for _ in range(3):
            ema(z)
        results.append(state(ema))
    for k in results[0]:
        assert torch.equal(results[0][k], results[1][k]), k


def test_unused_codes_stay_finite_and_match_the_oracle(mv):
    """Latents near 8 of the 512 codes: the other 504 are divided by a tiny smoothed_j and move far away."""
    g = torch.Generator().manual_seed(11)
    E = trained_codebook(512, 64, 4)
    centres = E[:8]
    z = (centres[torch.randint(0, 8, (4 * 16 * 16,), generator=g)] + 0.01 * torch.randn(4 * 16 * 16, 64, generator=g))
    z = z.view(4, 16, 16, 64).permute(0, 3, 1, 2).contiguous()
    for trained in (False, True):
        ema, _ = pair(mv, E, trained_state=trained)
        for _ in range(3):
            pre = state(ema)
            _, _, _, idx = ema(z.cuda())
            assert int(torch.unique(idx).numel()) <= 8
            check_update(ema, pre, z, idx)


# ----------------------------------------------------------------------------------------------- what never updates
def test_eval_get_code_indices_and_extractor_change_nothing(mv):
    ema, _ = pair(mv, trained_codebook(512, 64, 5), trained_state=True)
    z = make_z(4, 64, 8, 8, 9).cuda()
    ema(z)                                                        # one update so that the state is not the initial one
    torch.cuda.synchronize()
    before = state(ema)
    ema.eval()
    ema(z)
    with torch.no_grad():
        ema(z)
    ema.get_code_indices(z)
    ema.get_codebook_usage_percentage(z)
    ex = mv.CodeExtractor(ema)
    ex.push(z)
    ex.finish()
    torch.cuda.synchronize()
    after = state(ema)
    for k in before:
        assert torch.equal(before[k], after[k]), k
    ema.train()
    with torch.no_grad():                                         # a training-mode forward updates even without grad
        ema(z)
    assert not torch.equal(state(ema)["cs"], after["cs"])


# ----------------------------------------------------------------------------------------------- gradients
def test_gradients_and_the_saved_codebook(mv):
    ema, _ = pair(mv, trained_codebook(512, 64, 6), trained_state=True)
    z = make_z(4, 64, 8, 8, 12).cuda()
    zc = z.clone().requires_grad_(True)
    q, commit, embed, idx = ema(zc)
    assert embed.requires_grad and float(embed) > 0
    assert torch.autograd.grad(embed, zc, retain_graph=True, allow_unused=True) == (None,)
    (q.sum() + commit + embed).backward()
    assert ema.embedding.weight.grad is None
    # two training forwards, then the first one's backward: its saved pre-update codebook was overwritten
    z1 = z.clone().requires_grad_(True)
    q1, c1, _, _ = ema(z1)
    ema(z.clone().requires_grad_(True))
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        (q1.sum() + c1).backward()


class _TinyEMANet(torch.nn.Module):
    def __init__(self, mv):
        super().__init__()
        nn = torch.nn
        self.encoder = nn.Sequential(nn.Conv2d(3, 16, 3, 2, 1), nn.LeakyReLU(), nn.Conv2d(16, 64, 3, 2, 1))
        self.vq_layer = mv.VectorQuantizerEMA(512, 64)
        self.decoder = nn.Sequential(nn.ConvTranspose2d(64, 16, 4, 2, 1), nn.LeakyReLU(), nn.ConvTranspose2d(16, 3, 4, 2, 1))

    def forward(self, x):
        enc = self.encoder(x)
        q, commit, embed, _ = self.vq_layer(enc)
        rec = self.decoder(q)
        return enc, [torch.nn.functional.mse_loss(rec, x), embed, 0.25 * commit]


def test_mtl_backward_in_a_model_equals_the_oracle_aggregation(mv):
    """k = 3 with embedding_loss among the objectives: its Jacobian row is the zero row, the segmented path builds no
    [k, P] matrix, and the shared parameters receive the oracle's UPGrad aggregation of the rows autograd gives."""
    from movae_b200 import autojac
    from oracle import aggregation as oa

    torch.manual_seed(0)
    net = _TinyEMANet(mv).cuda()
    x = (torch.rand(8, 3, 16, 16, generator=torch.Generator().manual_seed(5)) * 2 - 1).cuda()
    autojac._J_CACHE.clear()
    enc, losses = net(x)
    mv.mtl_backward(losses=losses, features=[enc], aggregator=mv.make_aggregator("upgrad"), retain_graph=True)
    torch.cuda.synchronize()
    assert not autojac._J_CACHE, "the segmented path must not allocate a Jacobian"
    shared = list(net.encoder.parameters())
    rows = []
    for loss in losses:
        (fg,) = torch.autograd.grad(loss, [enc], retain_graph=True, allow_unused=True)
        if fg is None:
            rows.append(torch.zeros(sum(p.numel() for p in shared)))
            continue
        gs = torch.autograd.grad(enc, shared, grad_outputs=fg, retain_graph=True)
        rows.append(torch.cat([g.reshape(-1) for g in gs]).cpu())
    assert torch.count_nonzero(rows[1]) == 0
    J = torch.stack(rows)
    _, _, g_ref, _ = oa.aggregate("upgrad", J)
    got = torch.cat([p.grad.reshape(-1) for p in shared]).cpu()
    np.testing.assert_allclose(got.numpy(), g_ref.numpy(), rtol=1e-4, atol=1e-6)
    dec_ref = torch.autograd.grad(losses[0], list(net.decoder.parameters()), retain_graph=True)
    for p, g in zip(net.decoder.parameters(), dec_ref):
        np.testing.assert_allclose(p.grad.cpu().numpy(), g.cpu().numpy(), rtol=1e-5, atol=1e-7)
    assert net.vq_layer.embedding.weight.grad is None


def test_graphed_train_step_equals_eager(mv):
    """Five GraphedStep replays of the whole train step (Adam) == five eager steps, bit for bit: parameters, codebook,
    cluster_size and embed_avg."""
    x = (torch.rand(8, 3, 16, 16, generator=torch.Generator().manual_seed(5)) * 2 - 1).cuda()
    nets = []
    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True                   # cuDNN may otherwise pick a non-deterministic wgrad algorithm
    try:
        _graphed_vs_eager(mv, x, nets)
    finally:
        torch.backends.cudnn.deterministic = det
    assert set(nets[0]) == set(nets[1])
    for n in nets[0]:
        assert torch.equal(nets[0][n], nets[1][n]), n


def _graphed_vs_eager(mv, x, nets):
    for graphed in (False, True):
        torch.manual_seed(0)
        net = _TinyEMANet(mv).cuda()
        opt = mv.make_optimizer("adam", net.parameters(), lr=1e-3)
        agg = mv.make_aggregator("upgrad")

        def step(net=net, opt=opt, agg=agg):
            opt.zero_grad()
            enc, losses = net(x)
            mv.mtl_backward(losses=losses, features=[enc], aggregator=agg, retain_graph=True)
            opt.step()

        warmup = 2
        if graphed:
            g = mv.GraphedStep(step, warmup=warmup)          # runs `warmup` eager steps, then captures
            for _ in range(5):
                g()
        else:
            for _ in range(warmup + 5):
                step()
        torch.cuda.synchronize()
        nets.append({**{n: p.detach().cpu().clone() for n, p in net.named_parameters()},
                     **{n: b.detach().cpu().clone() for n, b in net.named_buffers()}})


def test_stats_reducer_on_one_gpu(mv):
    """A reducer that doubles the statistics: the oracle update with doubled counts and sums, through the split path."""
    for K, D, shape in ((512, 64, (4, 16, 16)), (512, 64, (3, 7, 9)), (100, 48, (3, 5, 7))):
        B, H, W = shape
        ema, _ = pair(mv, trained_codebook(K, D, 8), trained_state=True)
        seen = []
        ema.stats_reducer = lambda t: (seen.append(tuple(t.shape)), t.mul_(2.0))
        z = make_z(B, D, H, W, 21)
        pre = state(ema)
        _, _, _, idx = ema(z.cuda())
        assert seen == [(K + K * D,)]
        check_update(ema, pre, z, idx, count_scale=2.0)


# ----------------------------------------------------------------------------------------------- two GPUs
def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _ema_worker(rank, world, port, out_dir):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import movae_b200
        from movae_b200 import parallel

        torch.manual_seed(0)
        ema = movae_b200.VectorQuantizerEMA(512, 64).to(dev)
        with torch.no_grad():
            ema.embedding.weight.copy_(trained_codebook(512, 64, 9))
            ema.embed_avg.copy_(ema.embedding.weight)
        parallel.install_codebook_allreduce(ema)
        for step in range(3):
            z = make_z(16, 64, 8, 8, 300 + step)
            ema(z[rank * 8:(rank + 1) * 8].to(dev))
        torch.cuda.synchronize()
        torch.save({n: t.detach().cpu() for n, t in ema.state_dict().items()}, os.path.join(out_dir, f"ema{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_batch_sharded_replicas_stay_identical(mv, tmp_path):
    import torch.multiprocessing as mp

    world = 2
    mp.spawn(_ema_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    parts = [torch.load(os.path.join(tmp_path, f"ema{r}.pt")) for r in range(world)]
    ema = mv.VectorQuantizerEMA(512, 64).cuda()
    with torch.no_grad():
        ema.embedding.weight.copy_(trained_codebook(512, 64, 9))
        ema.embed_avg.copy_(ema.embedding.weight)
    for step in range(3):
        ema(make_z(16, 64, 8, 8, 300 + step).cuda())
    tol = {"cluster_size": dict(rtol=1e-6), "embed_avg": dict(rtol=1e-4, atol=1e-8), "embedding.weight": dict(rtol=1e-4, atol=1e-6)}
    for n, t in ema.state_dict().items():
        assert torch.equal(parts[0][n], parts[1][n]), f"{n}: replicas diverged"
        np.testing.assert_allclose(parts[0][n].numpy(), t.cpu().numpy(), err_msg=n, **tol[n])
