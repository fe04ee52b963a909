"""GPU parity tests (run on the B200 with -m gpu): CUDA path through the C-ABI vs the CPU oracle.

Tolerances (BASELINE.json north_star): Gramian, weights and aggregated gradient within
rtol 1e-5 / atol 1e-6 of the float64-accumulated oracle.  MGDA weights: the reference's own loop
differs by up to 1.5e-4 between float32 and float64 (SURVEY App. C.3), so MGDA weights are held to
atol 2e-4 unless the iteration counts coincide, in which case the tight tolerance applies.
"""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6
GOLDEN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "aggregation_golden.json")))
LOSSES = [0.34, 1e-3, 2.5e-4, 0.17, 2.0]


def synthetic_J(k, P, seed, decades=1.0, zero_row=None, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    g0 = torch.randn(P, generator=g, device=device)
    rows = torch.randn(k, P, generator=g, device=device)
    s = torch.logspace(0, -decades, k, device=device)
    J = s[:, None] * (0.3 * g0[None, :] + (1 - 0.09) ** 0.5 * rows)
    if zero_row is not None:
        J[zero_row] = 0
    return J.contiguous()


def losses_for(k):
    return torch.tensor([LOSSES[i % len(LOSSES)] for i in range(k)], dtype=torch.float32)


@pytest.fixture(scope="module")
def mv():
    import movae_b200
    return movae_b200


@pytest.fixture(scope="module")
def oa():
    from oracle import aggregation
    return aggregation


# ------------------------------------------------------------------------------------------------ K1
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("P", [1, 3, 4, 5, 1023, 4096, 4099, 262144 + 3, 1 << 20])
def test_gram_matches_fp64_oracle(mv, oa, k, P):
    J = synthetic_J(k, P, 100 * k + P % 97)
    G = mv.ops.gram(J).cpu().numpy()
    ref = oa.gramian_fp64(J.cpu())
    np.testing.assert_allclose(G, ref, rtol=RTOL, atol=ATOL)
    np.testing.assert_array_equal(G, G.T)


@pytest.mark.parametrize("k,P", [(3, 2_448_064), (2, 1_701_888), (5, 2_448_064), (3, 651_392), (8, 1_000_003)])
def test_gram_model_sizes_padded_and_unpadded_layouts(mv, oa, k, P):
    J = synthetic_J(k, P, 7)
    ref = oa.gramian_fp64(J.cpu())
    np.testing.assert_allclose(mv.ops.gram(J).cpu().numpy(), ref, rtol=RTOL, atol=ATOL)
    ld = (P + 3) // 4 * 4 + 8                      # engine layout: padded rows, float4 path
    buf = torch.zeros(k, ld, device="cuda")
    buf[:, :P] = J
    np.testing.assert_allclose(mv.ops.gram(buf[:, :P]).cpu().numpy(), ref, rtol=RTOL, atol=ATOL)
    off = torch.zeros(k * P + 1, device="cuda")    # base pointer only 4-byte aligned: scalar path
    Jm = off[1:].view(k, P)
    Jm.copy_(J)
    np.testing.assert_allclose(mv.ops.gram(Jm).cpu().numpy(), ref, rtol=RTOL, atol=ATOL)


def test_gram_edge_rows(mv, oa):
    P = 50_001
    cases = {
        "zero_row": synthetic_J(3, P, 1, zero_row=1),
        "dup_rows": synthetic_J(3, P, 2)[[0, 0, 2]].contiguous(),
        "rank1": (torch.tensor([1.0, -2.0, 0.5, 3.0], device="cuda")[:, None] * torch.randn(P, device="cuda")[None]),
        "scaled_1e6": synthetic_J(4, P, 3) * torch.tensor([1e6, 1.0, 1e-3, 1e-6], device="cuda")[:, None],
        "heavy_tail": torch.distributions.StudentT(2.5).sample((3, P)).cuda(),
    }
    for tag, J in cases.items():
        J = J.contiguous()
        G = mv.ops.gram(J).cpu().numpy()
        ref = oa.gramian_fp64(J.cpu())
        scale = np.sqrt(np.outer(np.diag(ref), np.diag(ref)))     # |J_i||J_j|: atol relative to row norms
        assert np.all(np.abs(G - ref) <= RTOL * np.abs(ref) + 1e-6 * scale), tag
    assert float(mv.ops.gram(cases["zero_row"].contiguous())[1].abs().max()) == 0.0


def test_gram_deterministic_and_accumulate(mv):
    J = synthetic_J(3, 3_000_001, 5)
    a, b = mv.ops.gram(J), mv.ops.gram(J)
    assert torch.equal(a, b)
    acc = torch.zeros(3, 3, dtype=torch.float64, device="cuda")
    for c0 in range(0, J.shape[1], 1_000_000):     # column-chunked accumulation == P-sharding on one GPU
        mv.ops.gram(J[:, c0:c0 + 1_000_000], out=acc, accumulate=True)
    np.testing.assert_allclose(acc.cpu().numpy(), a.cpu().numpy(), rtol=1e-7)   # chunk boundaries regroup the float32 chains


def test_gram_full_size_against_cublas_fp64(mv):
    """BASELINE size (k=3, P=1e8): size-independent check against an independent float64 GEMM."""
    J = synthetic_J(3, 100_000_000, 1234)
    G = mv.ops.gram(J)
    ref = torch.zeros(3, 3, dtype=torch.float64, device="cuda")
    for c0 in range(0, J.shape[1], 25_000_000):
        blk = J[:, c0:c0 + 25_000_000].double()
        ref += blk @ blk.T
    np.testing.assert_allclose(G.cpu().numpy(), ref.cpu().numpy(), rtol=RTOL, atol=ATOL)
    ref32 = (J @ J.T).double()                     # what the reference computes on this GPU
    print("\n[report] k=3 P=1e8  new-vs-fp64 %.2e   reference-fp32-vs-fp64 %.2e" % (
        float(((G - ref) / ref).abs().max()), float(((ref32 - ref) / ref).abs().max())))


# ------------------------------------------------------------------------------------------------ K2
def _weights(mv, key, G64, losses):
    parts = key.split(":")
    if parts[0] == "nupgrad":
        w, d = mv.ops.solve_upgrad(G64, None, 1e-4, 1e-4, "min_l2")
    elif parts[0] == "pnupgrad":
        w, d = mv.ops.solve_upgrad(G64, None, 1e-4, 1e-4, parts[1])
    elif parts[0] == "aligned_mtl":
        w, d = mv.ops.solve_aligned_mtl(G64, parts[1], None)
    else:
        stable = len(parts) == 3
        w, d = mv.ops.solve_mgda(G64, parts[1], losses, 1e-5, 250, stable, 1e-3 if stable else 1e-10)
    return w.cpu().numpy(), d.cpu().numpy()


@pytest.mark.parametrize("case", GOLDEN["cases"], ids=lambda c: c["tag"])
def test_solves_match_reference_golden(mv, case):
    from movae_b200 import _lib as L
    G64 = torch.tensor(case["G"], dtype=torch.float64, device="cuda")
    losses = torch.tensor(case["losses"], dtype=torch.float32, device="cuda")
    for key, exp in case["out"].items():
        w, d = _weights(mv, key, G64, losses)
        ew = np.array(exp["w"], dtype=np.float32)
        if key.startswith(("nupgrad", "pnupgrad")):
            # reference normalisation + wrapper code (nupgrad.py / pnupgrad.py) with the oracle's exact QP behind it
            np.testing.assert_allclose(w, ew, rtol=RTOL, atol=ATOL, err_msg=f"{case['tag']} {key}")
            assert d[L.DIAG_STATUS] == 0.0
        elif key.startswith("aligned_mtl"):
            # golden = the reference's float32 eigh; it is itself eps32*cond(G) away from the float64
            # arbiter (SURVEY App. C.4: 5e-6 at k=8 tier A, 1e-4 at cond 1e4) -> scaled tolerance here,
            # the tight rtol 1e-5 gate is against the float64 arbiter in test_whole_step_matches_oracle
            tol = (5e-4 if case["tag"] == "tierB_k3" else 3e-5) * float(np.abs(ew).max())
            np.testing.assert_allclose(w, ew, rtol=0, atol=tol, err_msg=f"{case['tag']} {key}")
        else:
            same_path = int(d[L.DIAG_COUNT]) == exp["convergence_count"]
            if same_path and "stable" not in key:
                np.testing.assert_allclose(w, ew, rtol=2e-5, atol=2e-6, err_msg=f"{case['tag']} {key}")
                # the exit gamma (< epsilon) is a cancellation-dominated quantity: only its side of epsilon is stable
                if exp["gamma"] < 1e-5:
                    assert d[L.DIAG_GAMMA] < 1e-5
                else:
                    assert d[L.DIAG_GAMMA] == pytest.approx(exp["gamma"], rel=1e-3)
            else:
                np.testing.assert_allclose(w, ew, rtol=0, atol=2e-4, err_msg=f"{case['tag']} {key}")


@pytest.mark.parametrize("k", [2, 3, 4, 5, 8])
@pytest.mark.parametrize("variant", ["tierA", "zero_row", "tierB", "pref"])
def test_upgrad_weights_match_oracle(mv, oa, k, variant):
    from movae_b200 import _lib as L
    J = synthetic_J(k, 4099, 40 + k, decades=2.0 if variant == "tierB" else 1.0,
                    zero_row=1 if variant == "zero_row" else None).cpu()
    G32 = oa.arbiter_gramian(J)
    pref = torch.linspace(0.5, 1.5, k) if variant == "pref" else None
    w_ref = oa.upgrad_weights(G32, pref_vector=pref).numpy()
    w, d = mv.ops.solve_upgrad(G32.double().cuda(), pref, 1e-4, 1e-4)
    np.testing.assert_allclose(w.cpu().numpy(), w_ref, rtol=RTOL, atol=ATOL)
    d = d.cpu().numpy()
    assert d[L.DIAG_STATUS] == 0.0 and d[L.DIAG_RESIDUAL] < 1e-12


def test_upgrad_docstring_kat_and_zero_gramian(mv):
    J = torch.tensor([[-4.0, 1.0, 1.0], [6.0, 1.0, 1.0]], device="cuda")
    g = mv.UPGrad()(J)
    np.testing.assert_allclose(g.cpu().numpy(), [0.2929, 1.9004, 1.9004], atol=5e-5)    # nupgrad.py:55-62
    w, _ = mv.ops.solve_upgrad(torch.zeros(3, 3, dtype=torch.float64, device="cuda"), None, 1e-4, 1e-4)
    np.testing.assert_allclose(w.cpu().numpy(), np.full(3, 1 / 3), rtol=1e-6)


def test_docstring_kats_through_aggregators(mv):
    J = torch.tensor([[-4.0, 1.0, 1.0], [6.0, 1.0, 1.0]], device="cuda")
    ls = torch.tensor([0.5, 2.0], device="cuda")
    np.testing.assert_allclose(mv.MGDA()(J).cpu().numpy(), [0, 1, 1], atol=1e-6)                    # mgda.py:57-60
    np.testing.assert_allclose(mv.MGDA("l2")(J).cpu().numpy(), [1, 1, 1], atol=1e-6)                # mgda.py:65-68
    a = mv.MGDA("loss"); a.set_losses(ls)
    np.testing.assert_allclose(a(J).cpu().numpy(), [3.4900, 1, 1], atol=5e-5)                       # mgda.py:73-77
    assert a.mgda_weighting.convergence_count == 2
    a = mv.MGDA("loss+"); a.set_losses(ls)
    np.testing.assert_allclose(a(J).cpu().numpy(), [4.1606, 1, 1], atol=5e-5)                       # mgda.py:82-86
    np.testing.assert_allclose(mv.AlignedMTL()(J).cpu().numpy(), [0.2133, 0.9673, 0.9673], atol=5e-5)
    np.testing.assert_allclose(mv.AlignedMTL(scale_mode="rmse")(J).cpu().numpy(), [0.5764, 2.6142, 2.6142], atol=5e-5)
    np.testing.assert_allclose(mv.Sum()(J).cpu().numpy(), [2, 2, 2], atol=0)
    np.testing.assert_allclose(mv.Mean()(J).cpu().numpy(), [1, 1, 1], atol=0)
    Jz = torch.tensor([[-4.0, 1.0, 1.0], [0.0, 0.0, 0.0], [6.0, 1.0, 1.0]], device="cuda")
    amtl = mv.AlignedMTL()
    np.testing.assert_allclose(amtl(Jz).cpu().numpy(), [0.1422, 0.6449, 0.6449], atol=5e-5)         # SURVEY 8c
    assert amtl.weighting.rank == 2
    m = mv.MGDA("l2")
    assert float(m(Jz).abs().max()) == 0.0 and m.mgda_weighting.convergence_count in (2, 3)


def test_mgda_vertex_fixpoint_reports_max_iters(mv, oa):
    """Dominated-vertex case (SURVEY App. C.3): the reference spins to max_iters with gamma == 1."""
    G = torch.tensor([[1.0, 2.0, 2.0], [2.0, 100.0, 50.0], [2.0, 50.0, 100.0]])
    w_ref, count, gamma = oa.mgda_weights(G)
    assert count == 250 and gamma == 1.0
    from movae_b200 import _lib as L
    w, d = mv.ops.solve_mgda(G.double().cuda(), "none", None, 1e-5, 250, False, 1e-10)
    d = d.cpu().numpy()
    np.testing.assert_allclose(w.cpu().numpy(), w_ref.numpy(), atol=0)
    assert int(d[L.DIAG_COUNT]) == 250 and d[L.DIAG_GAMMA] == 1.0


# ------------------------------------------------------------------------------------------------ K3 + whole step
@pytest.mark.parametrize("k,P", [(1, 5), (2, 1023), (3, 4099), (3, 2_448_064), (5, 1_000_003), (8, 262_147)])
def test_recombine_matches_fp64_oracle(mv, oa, k, P):
    J = synthetic_J(k, P, 11)
    w = torch.linspace(-0.7, 1.3, k, device="cuda")
    ref = oa.recombine_fp64(w.cpu(), J.cpu()).numpy()
    np.testing.assert_allclose(mv.ops.recombine(J, w).cpu().numpy(), ref, rtol=RTOL, atol=ATOL)
    out = torch.ones(P, device="cuda")
    mv.ops.recombine(J, w, out=out, accumulate=True)
    np.testing.assert_allclose(out.cpu().numpy(), ref + 1.0, rtol=RTOL, atol=2 * ATOL)
    off = torch.zeros(k * P + 1, device="cuda")
    Jm = off[1:].view(k, P); Jm.copy_(J)
    np.testing.assert_allclose(mv.ops.recombine(Jm, w).cpu().numpy(), ref, rtol=RTOL, atol=ATOL)


AGGS = ["sum", "mean", "upgrad", "aligned_mtl", "aligned_mtl_median", "aligned_mtl_rmse", "mgda", "mgda_ln",
        "mgda_gn", "mgda_lgn"]


def _make(mv, name):
    return mv.Sum() if name == "sum" else mv.make_aggregator(name)


@pytest.mark.parametrize("name", AGGS)
@pytest.mark.parametrize("k,P,zero_row", [(2, 1_701_888, None), (3, 2_448_064, None), (3, 651_392, 1), (4, 300_001, None),
                                          (5, 300_001, None), (8, 100_003, None)])
def test_whole_step_matches_oracle(mv, oa, name, k, P, zero_row):
    J = synthetic_J(k, P, 1234 + k, zero_row=zero_row)
    losses = losses_for(k)
    agg = _make(mv, name)
    if isinstance(agg, mv.MGDA):
        agg.set_losses(losses.cuda())
    seen = {}
    agg.weighting.register_forward_hook(lambda m, inp, out: seen.update(J=inp[0], w=out))   # main.py:1248-1250
    g = agg(J)
    G_ref, w_ref, g_ref, info = oa.aggregate(name, J.cpu(), losses, amtl_dtype=torch.float64)
    assert seen["J"].shape == J.shape and seen["w"].shape == (k,)
    np.testing.assert_allclose(agg.weighting.last_gramian.cpu().numpy(), G_ref.double().numpy(), rtol=RTOL, atol=ATOL)
    w = seen["w"].cpu().numpy()
    if name.startswith("mgda"):
        same = agg.mgda_weighting.convergence_count == info["convergence_count"]
        wtol = dict(rtol=2e-5, atol=2e-6) if same else dict(rtol=0, atol=2e-4)
        np.testing.assert_allclose(w, w_ref.numpy(), **wtol)
        scale = float(J.abs().max()) * k
        np.testing.assert_allclose(g.cpu().numpy(), g_ref.numpy(), rtol=RTOL if same else 1e-3,
                                   atol=ATOL if same else 2e-4 * scale)
    else:
        np.testing.assert_allclose(w, w_ref.numpy(), rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(g.cpu().numpy(), g_ref.numpy(), rtol=RTOL, atol=ATOL)
    sim = oa.gradient_similarity_from_gramian(G_ref.double().numpy(), w_ref.tolist())
    assert agg.weighting.gradient_similarity == pytest.approx(sim, abs=1e-4)


def test_error_behaviour_on_gpu(mv):
    J = synthetic_J(3, 100, 0)
    with pytest.raises(RuntimeError):                       # mgda.py:326-330
        mv.MGDA("loss")(J)
    m = mv.MGDA("loss+"); m.set_losses(torch.ones(2, device="cuda"))
    with pytest.raises(ValueError):                         # mgda.py:357-361
        m(J)
    with pytest.raises(ValueError):                         # aligned_mtl.py:127-130
        mv.AlignedMTL(scale_mode="bogus")(J)
    with pytest.raises(TypeError):
        mv.UPGrad()(J.double())
    with pytest.raises(RuntimeError, match="CUDA|cuda"):
        mv.UPGrad()(torch.randn(9, 10, device="cuda"))


# ------------------------------------------------------------------------------------------------ engine
class _TinyMTL(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.enc = torch.nn.Sequential(torch.nn.Linear(7, 16), torch.nn.Tanh(), torch.nn.Linear(16, 5))
        self.h1 = torch.nn.Linear(5, 3)
        self.h2 = torch.nn.Linear(5, 1)
        self.code = torch.nn.Parameter(torch.randn(5))

    def forward(self, x):
        f = self.enc(x)
        l1 = self.h1(f).pow(2).mean()
        l2 = (self.h2(f) - 1).abs().mean()
        l3 = (self.code - f.detach().mean(0)).pow(2).mean()        # like embedding_loss: no shared-param dependence
        return f, [l1, l2, l3]


@pytest.fixture(params=["segmented", "flat_jacobian"])
def jacobian_mode(request, mv):
    """Makes the test's aggregators for one of the engine's two paths: the segmented launch over the gradient tensors
    (the default), or the flat J, forced by a forward hook on the weighting (hooks receive J).  `hooked` records the
    hook calls."""
    hooked = []

    def make(name):
        agg = mv.make_aggregator(name)
        if request.param == "flat_jacobian":
            agg.weighting.register_forward_hook(lambda m, inp, out: hooked.append(tuple(inp[0].shape)))
        return agg

    make.mode, make.hooked = request.param, hooked
    return make


@pytest.mark.parametrize("name", ["upgrad", "aligned_mtl", "mgda_ln"])
def test_mtl_backward_and_backward_match_oracle(mv, oa, name, jacobian_mode):
    make_aggregator = jacobian_mode
    torch.manual_seed(0)
    net = _TinyMTL().cuda()
    x = torch.randn(32, 7, device="cuda")
    # ---- expected, from plain autograd + oracle --------------------------------------------
    f, losses = net(x)
    shared = list(net.enc.parameters())
    rows = []
    for l in losses:
        gs = torch.autograd.grad(l, shared, retain_graph=True, allow_unused=True)
        rows.append(torch.cat([torch.zeros_like(p).flatten() if g is None else g.flatten() for p, g in zip(shared, gs)]))
    Jm = torch.stack(rows).cpu()
    _, _, g_ref, _ = oa.aggregate(name, Jm, amtl_dtype=torch.float64)
    head_ref = {n: torch.autograd.grad(sum(losses), p, retain_graph=True)[0] for n, p in
                [("h1", net.h1.weight), ("h2", net.h2.weight), ("code", net.code)]}
    # ---- mtl_backward ----------------------------------------------------------------------
    net.zero_grad(set_to_none=True)
    f, losses = net(x)
    mv.mtl_backward(losses=losses, features=[f], aggregator=make_aggregator(name), retain_graph=True)
    got = torch.cat([p.grad.flatten() for p in shared]).cpu()
    np.testing.assert_allclose(got.numpy(), g_ref.numpy(), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(net.h1.weight.grad.cpu().numpy(), head_ref["h1"].cpu().numpy(), rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(net.h2.weight.grad.cpu().numpy(), head_ref["h2"].cpu().numpy(), rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(net.code.grad.cpu().numpy(), head_ref["code"].cpu().numpy(), rtol=1e-5, atol=1e-7)
    # second call accumulates (torchjd Accumulate: += when .grad exists)
    f, losses = net(x)
    mv.mtl_backward(losses=losses, features=[f], aggregator=make_aggregator(name), retain_graph=True)
    got2 = torch.cat([p.grad.flatten() for p in shared]).cpu()
    np.testing.assert_allclose(got2.numpy(), 2 * g_ref.numpy(), rtol=RTOL, atol=2 * ATOL)
    # ---- backward over ALL parameters -------------------------------------------------------
    net.zero_grad(set_to_none=True)
    f, losses = net(x)
    params = [p for p in net.parameters()]
    rows = []
    for l in losses:
        gs = torch.autograd.grad(l, params, retain_graph=True, allow_unused=True)
        rows.append(torch.cat([torch.zeros_like(p).flatten() if g is None else g.flatten() for p, g in zip(params, gs)]))
    _, _, g_all, _ = oa.aggregate(name, torch.stack(rows).cpu(), amtl_dtype=torch.float64)
    mv.backward(losses, aggregator=make_aggregator(name), inputs=params)
    got = torch.cat([p.grad.flatten() for p in params]).cpu()
    np.testing.assert_allclose(got.numpy(), g_all.numpy(), rtol=RTOL, atol=ATOL)
    assert bool(jacobian_mode.hooked) == (jacobian_mode.mode == "flat_jacobian")      # the path under test ran


# ------------------------------------------------------------------------------------ 8f "next" aggregators
def test_nupgrad_pnupgrad_comfort_aggregators(mv, oa):
    J = synthetic_J(3, 50_001, 91)
    Jc = J.cpu()
    G32 = oa.arbiter_gramian(Jc)
    # NUPGrad
    g = mv.NUPGrad()(J)
    w_ref = oa.nupgrad_weights(G32, mode="min_l2")
    np.testing.assert_allclose(g.cpu().numpy(), oa.recombine_fp64(w_ref, Jc).numpy(), rtol=RTOL, atol=ATOL)
    # PNUPGrad: prob 1 -> always the cosine-normalised branch, prob 0 -> always NUPGrad's; the draw uses torch's host RNG
    for prob, mode in ((1.0, "l2"), (0.0, "min_l2")):
        agg = mv.PNUPGrad(prob=prob)
        g = agg(J)
        w_ref = oa.nupgrad_weights(G32, mode=mode)
        np.testing.assert_allclose(g.cpu().numpy(), oa.recombine_fp64(w_ref, Jc).numpy(), rtol=RTOL, atol=ATOL)
    torch.manual_seed(5)
    draws = [torch.rand(1).item() < 0.5 for _ in range(6)]
    torch.manual_seed(5)
    agg = mv.PNUPGrad(prob=0.5)
    seen = []
    for _ in range(6):
        agg(J)
        seen.append(agg.weighting._mode == "l2")
    assert seen == draws                                   # same RNG stream consumption as pnupgrad.py:129
    # COMFORT = (1 - beta) MGDA + beta UPGrad, one Gramian pass
    losses = torch.tensor([0.34, 1e-3, 2.5e-4], device="cuda")
    for epoch, total in ((1, 10), (4, 10), (10, 10)):
        c = mv.COMFORT(mgda_norm_type="loss+", mgda_min_eigenvalue_eps=1e-10)
        c.set_epoch(epoch, total)
        c.set_losses(losses)
        beta = oa.comfort_beta(epoch, total)
        assert mv.beta_schedule(epoch, total) == pytest.approx(beta, rel=1e-12)
        m = mv.MGDA(norm_type="loss+")
        m.set_losses(losses)
        ref = (1.0 - beta) * m(J) + beta * mv.UPGrad()(J)
        np.testing.assert_allclose(c(J).cpu().numpy(), ref.cpu().numpy(), rtol=2e-5, atol=2e-6)
    assert mv.beta_schedule(1, 10) == pytest.approx(0.01) and mv.beta_schedule(10, 10) == pytest.approx(1.0)
    assert isinstance(mv.make_aggregator("comfort"), mv.COMFORT) and isinstance(mv.make_aggregator("nupgrad"), mv.NUPGrad)
    hits = []
    c.weighting.register_forward_hook(lambda mod, inp, out: hits.append(out.shape))       # hook contract (main.py:1248-1250)
    c(J)
    assert hits == [torch.Size([3])]


def test_non_finite_jacobian_is_reported_not_hidden(mv):
    """A NaN in J (diverged training): torchjd's UPGrad raises ValueError when quadprog fails; here the solve flags it in
    last_diag[STATUS] and check_status() raises the same exception -- no crash, no hang, no silent success."""
    J = synthetic_J(3, 10_000, 5)
    J[1, 17] = float("nan")
    agg = mv.UPGrad()
    g = agg(J)
    torch.cuda.synchronize()
    assert not bool(torch.isfinite(g).all())
    with pytest.raises(ValueError):
        agg.weighting.check_status()
    for name in ("aligned_mtl", "mgda_ln", "sum"):
        a = mv.make_aggregator(name) if name != "sum" else mv.Sum()
        a(J)                                          # must terminate
    torch.cuda.synchronize()
    ok = mv.UPGrad()
    ok(synthetic_J(3, 10_000, 6))
    ok.weighting.check_status()                       # finite input: no exception


@pytest.mark.parametrize("k", [2, 3, 4, 5, 8])
@pytest.mark.parametrize("zero_row", [None, 1])
def test_dualproj_matches_oracle(mv, oa, k, zero_row):
    """torchjd DualProj (main.py:1221-1222) on the K2 enumeration: weights and aggregated gradient against the oracle."""
    J = synthetic_J(k, 20_003, 900 + k, zero_row=zero_row)
    J[0] = -0.6 * J[k - 1] + 0.2 * J[0]                                   # conflict: some bounds become active
    agg = mv.make_aggregator("dualproj")
    assert isinstance(agg, mv.DualProj)
    g = agg(J)
    w = agg.weighting(J)
    G32 = torch.from_numpy(oa.gramian_fp64(J.cpu())).to(torch.float32)
    w_ref = oa.dualproj_weights(G32)
    np.testing.assert_allclose(w.cpu().numpy(), w_ref.numpy(), rtol=RTOL, atol=ATOL)
    g_ref = oa.recombine_fp64(w_ref, J.cpu())
    np.testing.assert_allclose(g.cpu().numpy(), g_ref.numpy(), rtol=RTOL, atol=ATOL)
    agg.weighting.check_status()
