"""GPU tests of the PCGrad and IMTL-G aggregators (MOVAE_SOLVE_PCGRAD / MOVAE_SOLVE_IMTLG, solved inside the fused
aggregation launch) against the CPU oracles of tests/oracle_pcgrad_imtlg.py: parity, every launch path, CUDA-graph replay
of PCGrad's host draw, hooks, non-finite input, and (2 GPUs) the replicated draw of the P-sharded and data-parallel paths.

Tolerances: rtol 1e-5 / atol 1e-6.  PCGrad is held to torchjd's float32 loop on the arbiter Gramian under the same
permutations (the seed is reset before the oracle draws them); IMTL-G to the float64 eigen-decomposition arbiter."""
import os
import socket

import numpy as np
import pytest
import torch

import oracle_pcgrad_imtlg as op

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6
NAMES = ("pcgrad", "imtlg")


@pytest.fixture(scope="module")
def mv():
    import movae_b200
    return movae_b200


@pytest.fixture(scope="module")
def oa():
    from oracle import aggregation
    return aggregation


def make_J(k, P, seed, case="random", device="cuda"):
    """`random`: rows of alternating sign around a shared component (conflicting pairs for PCGrad to project);
    `zero_row`: row 1 identically zero; `conflict`: row 1 = -0.5 row 0 + noise; `disjoint`: row i supported on its own
    column block (exactly orthogonal); `duplicate`: row 1 = row 0."""
    g = torch.Generator(device=device).manual_seed(seed)
    g0 = torch.randn(P, generator=g, device=device)
    rows = torch.randn(k, P, generator=g, device=device)
    s = torch.logspace(0, -1, k, device=device) * torch.tensor([(-1.0) ** i for i in range(k)], device=device)
    J = s[:, None] * (0.3 * g0[None, :] + 0.91 ** 0.5 * rows)
    if case == "zero_row" and k > 1:
        J[1] = 0
    elif case == "conflict" and k > 1:
        J[1] = -0.5 * J[0] + 0.1 * rows[1]
    elif case == "disjoint":
        mask = torch.zeros(k, P, device=device)
        for i in range(k):
            mask[i, i * (P // k):(i + 1) * (P // k)] = 1
        J = J * mask
    elif case == "duplicate" and k > 1:
        J[1] = J[0]
    return J.contiguous()


def reference_weights(oa, name, J, seed):
    """The oracle's weights on the arbiter Gramian; PCGrad draws its permutations from the host RNG reset to `seed`."""
    G32 = oa.arbiter_gramian(J.cpu())
    if name == "pcgrad":
        torch.manual_seed(seed)
        return op.pcgrad_weights(G32, op.draw_permutations(J.shape[0]))
    return op.imtlg_weights_fp64(G32)[0]


# ------------------------------------------------------------------------------------------------------------ parity
def _check_step(mv, oa, name, J, seed):
    k = J.shape[0]
    agg = mv.make_aggregator(name)
    out = torch.full((J.shape[1],), 3.0, device="cuda")
    torch.manual_seed(seed)
    w = agg.aggregate_into(J, out)
    agg.weighting.check_status()
    np.testing.assert_allclose(agg.weighting.last_gramian.cpu().numpy(), oa.gramian_fp64(J.cpu()), rtol=RTOL, atol=ATOL)
    w_ref = reference_weights(oa, name, J, seed)
    np.testing.assert_allclose(w.cpu().numpy(), w_ref.numpy(), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(out.cpu().numpy(), oa.recombine_fp64(w.cpu(), J.cpu()).numpy(), rtol=RTOL, atol=ATOL)
    return agg, w


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("P", [4099, 1 << 20, 2_448_064])
def test_weights_and_gradient_match_oracle(mv, oa, name, k, P):
    _check_step(mv, oa, name, make_J(k, P, 97 * k + P % 89), seed=k)


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("k", [2, 3, 5, 8])
@pytest.mark.parametrize("case", ["zero_row", "conflict", "disjoint", "duplicate"])
def test_structured_jacobians(mv, oa, name, k, case):
    J = make_J(k, 1 << 20, 11 * k, case)
    agg, w = _check_step(mv, oa, name, J, seed=5)
    if name == "pcgrad" and case == "disjoint":
        assert torch.equal(w.cpu(), torch.ones(k))                 # orthogonal rows: nothing to project
    if name == "imtlg":
        _, rank = op.imtlg_weights_fp64(oa.arbiter_gramian(J.cpu()))
        assert agg.weighting.rank == rank == (k - 1 if case in ("zero_row", "duplicate") else k)
        if case != "duplicate":                                    # float32 pinv sits right at its tolerance on exact duplicates
            np.testing.assert_allclose(w.cpu().numpy(), op.imtlg_weights(oa.arbiter_gramian(J.cpu())).numpy(), rtol=1e-4, atol=1e-5)


def test_known_answers_on_the_device(mv):
    J = torch.tensor([[-4.0, 1.0, 1.0], [6.0, 1.0, 1.0]], device="cuda")
    np.testing.assert_allclose(mv.PCGrad()(J).cpu().numpy(), [0.5848, 3.8012, 3.8012], atol=5e-5)
    np.testing.assert_allclose(mv.IMTLG()(J).cpu().numpy(), [0.0767, 1.0000, 1.0000], atol=5e-5)
    np.testing.assert_allclose(mv.IMTLG().weighting(J).cpu().numpy(), [0.5923, 0.4077], atol=5e-5)
    w = mv.IMTLG().weighting(torch.zeros(3, 100, device="cuda"))
    assert torch.equal(w.cpu(), torch.zeros(3))                   # |sum(v)| < 1e-12 -> zeros


# ------------------------------------------------------------------------------------------------ every path agrees
class _TinyNet(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.enc = torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3, 2, 1), torch.nn.LeakyReLU(), torch.nn.Conv2d(8, 6, 3, 2, 1))
        self.h1 = torch.nn.Conv2d(6, 3, 1)
        self.h2 = torch.nn.Linear(6, 1)

    def forward(self, x):
        f = self.enc(x)
        return f, [self.h1(f).pow(2).mean(), -(self.h2(f.mean((2, 3))) - 1).abs().mean(), (f - 0.5).pow(2).mean()]


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("k", [3, 8])
def test_fused_segmented_standalone_and_reducer_paths_agree(mv, oa, name, k):
    sizes = [27, 130, 65_537, 300_000, 1_048_576 + 3]
    J = make_J(k, sum(sizes), 3 * k)
    rows, offs, off, c0 = [[] for _ in range(k)], [], 0, 0
    for n in sizes:
        for i in range(k):
            rows[i].append(J[i, c0:c0 + n].clone())
        offs.append(off)
        off += (n + 3) // 4 * 4
        c0 += n
    w_ref = reference_weights(oa, name, J, seed=9)

    torch.manual_seed(9)
    fused = mv.make_aggregator(name)
    w_fused = fused.aggregate_into(J, torch.empty(J.shape[1], device="cuda"))
    G = fused.weighting.last_gramian.clone()

    torch.manual_seed(9)
    seg = mv.make_aggregator(name)
    assert seg.supports_segments()
    out = torch.zeros(off, device="cuda")
    w_seg = seg.aggregate_segments_into(rows, sizes, offs, out)

    torch.manual_seed(9)
    alone = mv.make_aggregator(name)
    alone.weighting.prepare_step(J.device, k)                    # the step's draw (PCGrad), then K2 on a given Gramian
    w_k2 = alone.weighting.from_gramian(G)

    torch.manual_seed(9)
    red = mv.make_aggregator(name)
    red.weighting.gramian_reducer = lambda G: None               # K1 -> reducer -> K2 -> K3
    g_red = red(J)
    torch.manual_seed(9)
    w_red = red.weighting(J)

    np.testing.assert_array_equal(w_k2.cpu().numpy(), w_fused.cpu().numpy())        # same solve on the same Gramian
    for w in (w_fused, w_seg, w_red):
        np.testing.assert_allclose(w.cpu().numpy(), w_ref.numpy(), rtol=RTOL, atol=ATOL)
    g_ref = oa.recombine_fp64(w_fused.cpu(), J.cpu()).numpy()
    got = torch.cat([out[o:o + n] for o, n in zip(offs, sizes)])
    np.testing.assert_allclose(got.cpu().numpy(), g_ref, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(g_red.cpu().numpy(), g_ref, rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("name", NAMES)
def test_mtl_backward_and_backward_segmented_equal_flat(mv, name):
    """mtl_backward / backward run the segmented launch (no [k, P] Jacobian); a forward hook on the weighting forces the
    flat-J path.  Both draw the same permutations under the same seed: same gradients."""
    from movae_b200 import autojac

    x = torch.randn(8, 3, 16, 16, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    for api in ("mtl_backward", "backward"):
        grads = {}
        for mode in ("segments", "flat"):
            torch.manual_seed(0)
            net = _TinyNet().cuda()
            agg = mv.make_aggregator(name)
            seen = []
            if mode == "flat":
                agg.weighting.register_forward_hook(lambda m, inp, out: seen.append(tuple(inp[0].shape)))
            autojac._J_CACHE.clear()
            f, losses = net(x)
            torch.manual_seed(42)
            if api == "mtl_backward":
                mv.mtl_backward(losses=losses, features=[f], aggregator=agg, retain_graph=True)
            else:
                mv.backward(losses, aggregator=agg, retain_graph=True)
            torch.cuda.synchronize()
            agg.weighting.check_status()
            if mode == "segments":
                assert not autojac._J_CACHE, "the segmented path must not allocate a Jacobian"
            else:
                assert len(seen) == 1 and seen[0][0] == 3
            grads[mode] = {n: p.grad.detach().clone() for n, p in net.named_parameters()}
        for n in grads["flat"]:
            np.testing.assert_allclose(grads["segments"][n].cpu().numpy(), grads["flat"][n].cpu().numpy(), rtol=1e-5, atol=1e-7,
                                       err_msg=f"{api}: {n}")


# ------------------------------------------------------------------------------------------------------ graph replay
@pytest.mark.parametrize("name", NAMES)
def test_graph_replay_follows_the_host_draws(mv, name):
    k, P = 4, 300_001
    J = make_J(k, P, 77)
    out = torch.zeros(P, device="cuda")
    agg = mv.make_aggregator(name)
    agg.aggregate_into(J, out)                                   # eager first: allocates PCGrad's device table
    step = mv.GraphedStep(lambda: agg.aggregate_into(J, out), warmup=1)
    torch.manual_seed(2024)
    replayed = []
    for _ in range(6):
        w = step()
        torch.cuda.synchronize()
        replayed.append((w.clone(), out.clone()))
    torch.manual_seed(2024)
    eager = mv.make_aggregator(name)
    out_e = torch.zeros(P, device="cuda")
    for w, g in replayed:
        w_e = eager.aggregate_into(J, out_e)
        torch.cuda.synchronize()
        assert torch.equal(w, w_e) and torch.equal(g, out_e)
    if name == "pcgrad":
        assert len({tuple(w.tolist()) for w, _ in replayed}) > 1  # the draws changed the weights between replays
        fresh = mv.PCGrad()
        with pytest.raises(RuntimeError, match="eagerly"):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fresh.aggregate_into(J, out)


# ------------------------------------------------------------------------------------------------ hooks, status
@pytest.mark.parametrize("name", NAMES)
def test_forward_hooks_fire_once_and_the_handover_does_not_draw(mv, name):
    k = 3
    J = make_J(k, 100_003, 8)
    agg = mv.make_aggregator(name)
    seen = []
    agg.weighting.register_forward_hook(lambda m, inp, out: seen.append((m, inp, out.clone())))
    torch.manual_seed(31)
    g = agg(J)
    after = torch.rand(1)
    torch.manual_seed(31)
    if name == "pcgrad":
        op.draw_permutations(k)
    assert torch.equal(after, torch.rand(1))                     # PCGrad: k randperm(k) calls per aggregation; IMTL-G: none
    assert len(seen) == 1 and seen[0][0] is agg.weighting and len(seen[0][1]) == 1 and seen[0][1][0].data_ptr() == J.data_ptr()
    np.testing.assert_allclose(g.cpu().numpy(), mv.ops.recombine(J, seen[0][2]).cpu().numpy(), rtol=0, atol=0)


@pytest.mark.parametrize("name", NAMES)
def test_non_finite_jacobian_raises_on_check_status(mv, name):
    J = make_J(3, 10_000, 5)
    J[1, 17] = float("nan")
    agg = mv.make_aggregator(name)
    agg(J)
    with pytest.raises(ValueError):
        agg.weighting.check_status()
    ok = mv.make_aggregator(name)
    ok(make_J(3, 10_000, 6))
    ok.weighting.check_status()


def test_pcgrad_rejects_a_missing_or_corrupt_permutation_table(mv):
    from movae_b200 import _lib as L

    G = mv.ops.gram(make_J(3, 4099, 1))
    spec = L.SolveSpec(kind=L.SOLVE_PCGRAD)
    with pytest.raises(ValueError, match="permutation table"):
        mv.ops.solve(G, spec, None, None)
    good = torch.tensor([0, 1, 2, 2, 0, 1, 1, 2, 0], dtype=torch.float32, device="cuda")
    w, diag = mv.ops.solve(G, spec, None, good)
    assert float(diag[L.DIAG_STATUS]) == 0.0 and bool(torch.isfinite(w).all())
    for bad in ([0, 1, 2, 2, 0, 1, 1, 1, 0], [0, 1, 3, 2, 0, 1, 1, 2, 0], [0, 1, 2, 2, 0, 1, 1, 2, 0.5], [0, 1, -1, 2, 0, 1, 1, 2, 0]):
        w, diag = mv.ops.solve(G, spec, None, torch.tensor(bad, dtype=torch.float32, device="cuda"))
        assert float(diag[L.DIAG_STATUS]) == 1.0 and bool(torch.isnan(w).all()), bad


# ------------------------------------------------------------------------------------------------------ two GPUs
def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _cpu_J(k, P, seed=7):
    g = torch.Generator().manual_seed(seed)
    s = torch.logspace(0, -1, k) * torch.tensor([(-1.0) ** i for i in range(k)])
    return s[:, None] * (0.3 * torch.randn(P, generator=g)[None] + 0.91 ** 0.5 * torch.randn(k, P, generator=g))


def _multi_worker(rank, world, port, k, P, out_dir):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import movae_b200
        from movae_b200 import parallel

        J = _cpu_J(k, P)
        lo, hi = parallel.shard_columns(P, rank, world)
        Jl = J[:, lo:hi].contiguous().to(dev)
        res = {}
        for name in NAMES:
            torch.manual_seed(100 + rank)                       # different host RNGs: rank 0's draw must win everywhere
            agg = movae_b200.make_aggregator(name)
            ex = parallel.install_p2p_gramian_exchange(agg, dev)
            res[f"{name}:p2p"] = [agg.aggregate_into(Jl, torch.empty(hi - lo, device=dev)).cpu() for _ in range(3)]
            torch.cuda.synchronize()
            dist.barrier()
            ex.close()
            torch.manual_seed(100 + rank)
            agg = movae_b200.make_aggregator(name)
            dp = parallel.DataParallel(agg)                      # every rank holds the same Jacobian: the average is J
            Pp = dp.padded_columns(P)
            Jp = torch.zeros(k, Pp, device=dev)
            Jp[:, :P] = J.to(dev)
            out = torch.empty(P, device=dev)
            res[f"{name}:dp"] = [dp.aggregate_into(Jp, P, out, accumulate=False).cpu() for _ in range(3)]
            torch.cuda.synchronize()
            dist.barrier()
            if dp.exchange is not None:
                dp.exchange.close()
        torch.save(res, os.path.join(out_dir, f"pi{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("k,P", [(3, 1_000_003), (8, 40_000)])
def test_sharded_and_data_parallel_use_rank0_draw(tmp_path, mv, k, P):
    import torch.multiprocessing as mp

    world = 2
    mp.spawn(_multi_worker, args=(world, _free_port(), k, P, str(tmp_path)), nprocs=world, join=True)
    parts = [torch.load(os.path.join(tmp_path, f"pi{r}.pt")) for r in range(world)]
    J = _cpu_J(k, P).cuda()
    for name in NAMES:
        for mode in ("p2p", "dp"):
            torch.manual_seed(100)                              # rank 0's RNG stream
            agg = mv.make_aggregator(name)
            refs = [agg.aggregate_into(J, torch.empty(P, device="cuda")).cpu() for _ in range(3)]
            for step, w_ref in enumerate(refs):
                key = f"{name}:{mode}"
                assert torch.equal(parts[0][key][step], parts[1][key][step]), f"{key} step {step}: ranks differ"
                np.testing.assert_allclose(parts[0][key][step].numpy(), w_ref.numpy(), rtol=RTOL, atol=ATOL, err_msg=key)
