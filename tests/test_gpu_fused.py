"""GPU tests of the fused aggregation launch (csrc/aggregate.cu: Gramian pass -> solve -> recombination in ONE
cooperative kernel) against the three separate kernels and the float64 oracle, of its CUDA-graph capture, and of the
per-step host state (COMFORT's beta, PNUPGrad's draw) that a captured launch reads from device memory."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6
LOSSES = [0.34, 1e-3, 2.5e-4, 0.17, 2.0]


def synthetic_J(k, P, seed, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    g0 = torch.randn(P, generator=g, device=device)
    rows = torch.randn(k, P, generator=g, device=device)
    s = torch.logspace(0, -1, k, device=device)
    return (s[:, None] * (0.3 * g0[None, :] + 0.91 ** 0.5 * rows)).contiguous()


@pytest.fixture(scope="module")
def mv():
    import movae_b200
    return movae_b200


@pytest.fixture(scope="module")
def oa():
    from oracle import aggregation
    return aggregation


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("P", [1, 5, 4099, 300_001, 2_448_064])
@pytest.mark.parametrize("name", ["upgrad", "aligned_mtl", "mgda_lgn"])
def test_fused_launch_equals_separate_kernels_and_oracle(mv, oa, k, P, name):
    J = synthetic_J(k, P, 31 * k + P % 89)
    losses = torch.tensor([LOSSES[i % 5] for i in range(k)], device="cuda")
    agg = mv.make_aggregator(name)
    if isinstance(agg, mv.MGDA):
        agg.set_losses(losses)
    out = torch.full((P,), 7.0, device="cuda")
    w = agg.aggregate_into(J, out)                                   # ONE launch
    G = agg.weighting.last_gramian.clone()
    np.testing.assert_allclose(G.cpu().numpy(), oa.gramian_fp64(J.cpu()), rtol=RTOL, atol=ATOL)
    # the separate kernels on the same Gramian: K2 alone must give the same weights, K3 alone the same gradient
    w_sep = agg.weighting.from_gramian(G)
    np.testing.assert_array_equal(w.cpu().numpy(), w_sep.cpu().numpy())
    g_sep = mv.ops.recombine(J, w_sep)
    np.testing.assert_array_equal(out.cpu().numpy(), g_sep.cpu().numpy())
    g_ref = oa.recombine_fp64(w.cpu(), J.cpu())
    np.testing.assert_allclose(out.cpu().numpy(), g_ref.numpy(), rtol=RTOL, atol=ATOL)
    assert float(agg.weighting.last_diag[4]) == 0.0
    # accumulate mode adds to what is there
    w2 = agg.aggregate_into(J, out, accumulate=True)
    np.testing.assert_array_equal(w2.cpu().numpy(), w.cpu().numpy())
    np.testing.assert_allclose(out.cpu().numpy(), 2.0 * g_sep.cpu().numpy(), rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("k,P", [(3, 100_003), (8, 40_001)])
def test_fused_launch_scalar_path_for_unaligned_layouts(mv, oa, k, P):
    buf = torch.zeros(k * P + 1, device="cuda")
    Jm = buf[1:].view(k, P)                                          # base pointer only 4-byte aligned
    Jm.copy_(synthetic_J(k, P, 3))
    obuf = torch.zeros(P + 1, device="cuda")
    agg = mv.UPGrad()
    w = agg.aggregate_into(Jm, obuf[1:])
    g_ref = oa.recombine_fp64(w.cpu(), Jm.cpu())
    np.testing.assert_allclose(obuf[1:].cpu().numpy(), g_ref.numpy(), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(agg.weighting.last_gramian.cpu().numpy(), oa.gramian_fp64(Jm.cpu()), rtol=RTOL, atol=ATOL)


def test_fused_launch_is_bit_reproducible_and_reports_phase_times(mv):
    J = synthetic_J(3, 5_000_000, 11)
    agg = mv.UPGrad()
    a = agg(J).clone()
    Ga = agg.weighting.last_gramian.clone()
    for _ in range(3):
        b = agg(J)
        assert torch.equal(a, b) and torch.equal(Ga, agg.weighting.last_gramian)
    t_gram, t_solve, t_rec = mv.ops.aggregate_phase_times(mv.ops.current_workspace(J.device, 3))
    assert 0.0 < t_gram < 5.0 and 0.0 < t_solve < 5.0 and 0.0 < t_rec < 5.0      # ms, from the kernel's globaltimer stamps


def test_weighting_alone_is_one_launch_without_recombination_and_fires_hooks(mv, oa):
    J = synthetic_J(4, 123_457, 5)
    agg = mv.make_aggregator("aligned_mtl")
    seen = []
    agg.weighting.register_forward_hook(lambda m, inp, out: seen.append((inp[0].data_ptr(), out.clone())))
    w = agg.weighting(J)                                             # what a torchjd-style caller / the hooks use
    g = agg(J)
    assert len(seen) == 2 and seen[0][0] == J.data_ptr() and seen[1][0] == J.data_ptr()
    assert torch.equal(seen[0][1], seen[1][1]) and torch.equal(w, seen[0][1])
    np.testing.assert_allclose(g.cpu().numpy(), oa.recombine_fp64(w.cpu(), J.cpu()).numpy(), rtol=RTOL, atol=ATOL)


def test_fused_step_replays_from_a_cuda_graph(mv, oa):
    k, P = 3, 1_000_003
    J = synthetic_J(k, P, 21)
    out = torch.zeros(P, device="cuda")
    agg = mv.UPGrad()
    step = mv.GraphedStep(lambda: agg.aggregate_into(J, out), warmup=2)
    for seed in (22, 23):
        J.copy_(synthetic_J(k, P, seed))                             # new contents, same addresses
        w = step()
        torch.cuda.synchronize()
        eager = mv.UPGrad()
        g = eager(J)
        assert torch.equal(w, eager.weighting(J)) and torch.equal(out, g)
        np.testing.assert_allclose(out.cpu().numpy(), oa.recombine_fp64(w.cpu(), J.cpu()).numpy(), rtol=RTOL, atol=ATOL)


def test_comfort_beta_follows_set_epoch_after_capture(mv):
    """ADVICE r1: beta used to be a Python float folded in at capture; it now lives in device memory."""
    J = synthetic_J(3, 200_001, 41)
    losses = torch.tensor(LOSSES[:3], device="cuda")
    c = mv.COMFORT(mgda_norm_type="loss+", mgda_min_eigenvalue_eps=1e-10)
    c.set_losses(losses)
    c.set_epoch(1, 10)
    out = torch.zeros(J.shape[1], device="cuda")
    step = mv.GraphedStep(lambda: c.aggregate_into(J, out), warmup=2)
    m = mv.MGDA(norm_type="loss+")
    m.set_losses(losses)
    g_m, g_u = m(J).clone(), mv.UPGrad()(J).clone()
    seen = []
    for epoch in (1, 5, 10):
        c.set_epoch(epoch, 10)                                       # between steps, outside the graph
        step()
        torch.cuda.synchronize()
        beta = mv.beta_schedule(epoch, 10)
        ref = (1.0 - beta) * g_m + beta * g_u
        np.testing.assert_allclose(out.cpu().numpy(), ref.cpu().numpy(), rtol=2e-5, atol=2e-6)
        seen.append(out.clone())
    assert not torch.equal(seen[0], seen[2])


def test_pnupgrad_draws_once_per_replay_from_the_host_rng(mv, oa):
    J = synthetic_J(3, 50_001, 91)
    G32 = oa.arbiter_gramian(J.cpu())
    g_of = {m: oa.recombine_fp64(oa.nupgrad_weights(G32, mode=m), J.cpu()).numpy() for m in ("l2", "min_l2")}
    agg = mv.PNUPGrad(prob=0.5)
    out = torch.zeros(J.shape[1], device="cuda")
    agg.aggregate_into(J, out)                                       # eager first (allocates the device flag)
    step = mv.GraphedStep(lambda: agg.aggregate_into(J, out), warmup=1)
    torch.manual_seed(123)
    draws = ["l2" if torch.rand(1).item() < 0.5 else "min_l2" for _ in range(8)]
    assert len(set(draws)) == 2
    torch.manual_seed(123)
    for d in draws:
        step()
        torch.cuda.synchronize()
        assert agg.weighting._mode == d
        np.testing.assert_allclose(out.cpu().numpy(), g_of[d], rtol=RTOL, atol=ATOL)
    with pytest.raises(RuntimeError, match="GraphedStep"):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            agg.aggregate_into(J, out)


def test_status_is_checkable_on_every_weighting(mv):
    J = synthetic_J(3, 10_000, 5)
    J[1, 17] = float("nan")
    for name in ("upgrad", "aligned_mtl", "mgda_ln", "dualproj", "nupgrad"):
        agg = mv.make_aggregator(name)
        agg(J)
        with pytest.raises(ValueError):
            agg.weighting.check_status()


# ------------------------------------------------------------------------------------ segmented Jacobian (SURVEY 8f rank 1)
@pytest.mark.parametrize("k", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("name", ["upgrad", "aligned_mtl", "mgda_lgn", "comfort"])
def test_segmented_launch_equals_the_flat_jacobian(mv, oa, k, name):
    """movae_aggregate_segments_f32: the rows are separate tensors per segment (odd sizes, ragged tails, one tile-crossing
    segment, an identically zero row through a shared zero buffer) -- same Gramian, weights and gradient as the flat J, and
    bit for bit the gradient K3 computes from the same weights on J laid out like `out`."""
    sizes = [27, 4, 1, 130, 65_537, 300_000, 8, 1_048_576 + 3]
    g = torch.Generator(device="cuda").manual_seed(17 + k)
    scale = torch.logspace(0, -1, k, device="cuda")
    zero_row = 1 if k >= 3 else None
    zeros = torch.zeros(max(sizes), device="cuda")
    rows = [[(zeros if i == zero_row else scale[i] * torch.randn(n, generator=g, device="cuda")) for n in sizes] for i in range(k)]
    offs, off = [], 0
    for n in sizes:
        offs.append(off)
        off += (n + 3) // 4 * 4
    J = torch.cat([torch.stack([rows[i][s][:n] for i in range(k)]) for s, n in enumerate(sizes)], dim=1).contiguous()
    J_padded = torch.zeros(k, off, device="cuda")                   # each segment at its offset in `out`, zero columns between
    for s, (o, n) in enumerate(zip(offs, sizes)):
        J_padded[:, o:o + n] = torch.stack([rows[i][s][:n] for i in range(k)])
    losses = torch.tensor([LOSSES[i % 5] for i in range(k)], device="cuda")

    def make():
        a = mv.make_aggregator(name)
        if hasattr(a, "set_losses"):
            a.set_losses(losses)
        if name == "comfort":
            a.set_epoch(4, 10)
        return a
    agg = make()
    assert agg.supports_segments()
    out = torch.full((off,), 5.0, device="cuda")
    w = agg.aggregate_segments_into(rows, sizes, offs, out)
    ref = make()
    g_ref = ref(J)
    w_ref = ref.weighting(J) if name != "comfort" else ref.blended_weights(J)
    np.testing.assert_allclose(agg.weighting.last_gramian.cpu().numpy(), oa.gramian_fp64(J.cpu()), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(w.cpu().numpy(), w_ref.cpu().numpy(), rtol=2e-6, atol=2e-7)
    got = torch.cat([out[o:o + n] for o, n in zip(offs, sizes)])
    np.testing.assert_allclose(got.cpu().numpy(), g_ref.cpu().numpy(), rtol=RTOL, atol=ATOL)
    pad = torch.ones(off, dtype=torch.bool, device="cuda")
    for o, n in zip(offs, sizes):
        pad[o:o + n] = False
    assert bool((out[pad] == 5.0).all())                     # padding columns are never written
    assert torch.equal(out[~pad], mv.ops.recombine(J_padded, w)[~pad])
    before = out.clone()
    w2 = agg.aggregate_segments_into(rows, sizes, offs, out, accumulate=True)
    got2 = torch.cat([out[o:o + n] for o, n in zip(offs, sizes)])
    np.testing.assert_allclose(got2.cpu().numpy(), 2.0 * torch.cat([before[o:o + n] for o, n in zip(offs, sizes)]).cpu().numpy(), rtol=1e-6, atol=1e-7)
    assert torch.equal(out[~pad], mv.ops.recombine(J_padded, w2, out=before.clone(), accumulate=True)[~pad])


class _TinyNet(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.enc = torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3, 2, 1), torch.nn.LeakyReLU(), torch.nn.Conv2d(8, 6, 3, 2, 1))
        self.h1 = torch.nn.Conv2d(6, 3, 1)
        self.h2 = torch.nn.Linear(6, 1)

    def forward(self, x):
        f = self.enc(x)
        return f, [self.h1(f).pow(2).mean(), (self.h2(f.mean((2, 3))) - 1).abs().mean(), f.detach().pow(2).mean() * self.h2.bias.sum()]


@pytest.mark.parametrize("flat_params", [False, True])
def test_mtl_backward_builds_no_jacobian_and_copies_nothing(mv, monkeypatch, flat_params):
    """SURVEY 8f rank 1 / VERDICT r1 #6: the k backward passes' outputs ARE the Jacobian rows -- no [k, P] buffer, no
    multi-tensor copy; the result equals the flat-J path (forced by a forward hook on the weighting, which must see J)."""
    from movae_b200 import autojac

    torch.manual_seed(3)
    x = torch.randn(8, 3, 16, 16, device="cuda")
    grads = {}
    for mode in ("segments", "flat"):
        torch.manual_seed(0)
        net = _TinyNet().cuda()
        opt = mv.SGD(net.parameters(), lr=0.0) if flat_params else None
        agg = mv.make_aggregator("upgrad")
        seen = []
        if mode == "flat":
            agg.weighting.register_forward_hook(lambda m, inp, out: seen.append(tuple(inp[0].shape)))
        autojac._J_CACHE.clear()
        calls = []
        real = torch._foreach_copy_
        monkeypatch.setattr(torch, "_foreach_copy_", lambda *a, **k: (calls.append(sum(t.numel() for t in a[0])), real(*a, **k))[1])
        p_shared = sum(p.numel() for p in net.enc.parameters())
        f, losses = net(x)
        mv.mtl_backward(losses=losses, features=[f], aggregator=agg, retain_graph=True)
        monkeypatch.setattr(torch, "_foreach_copy_", real)
        torch.cuda.synchronize()
        if mode == "segments":
            # (with flat parameters the TASK-specific gradients of the heads are still adopted into the flat buffer by one
            # small multi-tensor copy; no copy may be as large as a Jacobian row)
            assert all(c < p_shared for c in calls) and not autojac._J_CACHE, "the segmented path must not copy the rows or allocate a Jacobian"
        else:
            assert any(c >= p_shared for c in calls) and autojac._J_CACHE and len(seen) == 1 and seen[0][0] == 3
        grads[mode] = {n: p.grad.detach().clone() for n, p in net.named_parameters()}
        del opt
    for n in grads["flat"]:
        np.testing.assert_allclose(grads["segments"][n].cpu().numpy(), grads["flat"][n].cpu().numpy(), rtol=1e-5, atol=1e-7, err_msg=n)


# ------------------------------------------------------------------------------------ host-buffer pipeline (bench `e2e`)
@pytest.mark.parametrize("name,k,P", [("upgrad", 3, 1_000_003), ("aligned_mtl", 2, 300_001), ("comfort", 4, 50_000)])
def test_host_plan_synchronous_and_pipelined_match_the_resident_path(mv, oa, name, k, P):
    """HostAggregationPlan: Jacobians in pinned HOST memory streamed through K1 / solve / K3 in column chunks; `run` is
    synchronous, `run_async` keeps two steps in flight (step i's D2H overlaps step i + 1's H2D).  Both must deliver, per
    step, the aggregated gradient of THAT step's Jacobian."""
    Js = [synthetic_J(k, P, 300 + i).cpu().pin_memory() for i in range(5)]
    agg = mv.make_aggregator(name)
    refs = [mv.make_aggregator(name)(J.cuda()).cpu() for J in Js]
    plan = mv.HostAggregationPlan(k, P, torch.device("cuda"), chunk_cols=1 << 16, depth=2)
    out = torch.empty(P, dtype=torch.float32).pin_memory()
    plan.run(Js[0], agg, out)
    np.testing.assert_allclose(out.numpy(), refs[0].numpy(), rtol=RTOL, atol=ATOL)
    outs = [torch.empty(P, dtype=torch.float32).pin_memory() for _ in Js]
    for J, o in zip(Js, outs):
        plan.run_async(J, agg, o)
    plan.wait()
    for o, r in zip(outs, refs):
        np.testing.assert_allclose(o.numpy(), r.numpy(), rtol=RTOL, atol=ATOL)
    with pytest.raises(ValueError):
        plan.run(Js[0].cuda(), agg, out)
