"""GPU parity tests of the VQ quantizer path (K4 tcgen05 search + exact re-check, K5 gather/loss/STE,
K6 backward) against the CPU oracle (oracle/vq.py, a restatement of the reference's
models/vq_vae.py:27-64 pinned to golden outputs of the reference module) -- all through the C ABI.

Parity bar (BASELINE.json north_star): code indices bit-exact except on "fp32 distance ties" (rows
whose two best codes are closer than 8 float32 ulps of the distance magnitude, where the reference's
own result depends on its BLAS accumulation order) -- those are counted and reported; quantized
output bit-exact where the index agrees; losses / gradients within rtol 1e-5 / atol 1e-6 unless noted.
"""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden import load_vq_golden  # noqa: E402

pytestmark = pytest.mark.gpu

GOLD = load_vq_golden()
TAGS = ("init", "trained", "dup")


@pytest.fixture(scope="module")
def mv():
    import movae_b200
    return movae_b200


@pytest.fixture(scope="module")
def ov():
    from oracle import vq
    return vq


def make_inputs(B, D, H, W, K, codebook, seed):
    g = torch.Generator().manual_seed(seed)
    z = 0.5 * torch.randn(B, D, H, W, generator=g)
    if codebook == "init":
        E = (torch.rand(K, D, generator=g) * 2 - 1) / K          # reference init U(-1/K, 1/K), vq_vae.py:25
    else:
        E = 0.5 * torch.randn(K, D, generator=g)
    return z, E


def _rows(x):
    """[B, D, H, W] -> [N, D] in the reference's row order (vq_vae.py:28-31)."""
    return np.ascontiguousarray(np.transpose(x, (0, 2, 3, 1))).reshape(-1, x.shape[1])


def _agreeing(mism, idx, idx_ref, K):
    """(rows whose index agrees, codes no disagreeing row touches): what stays comparable when fp32-tie rows differ."""
    ok = ~mism
    codes_ok = np.ones(K, dtype=bool)
    codes_ok[idx[mism]] = False
    codes_ok[idx_ref[mism]] = False
    return ok, codes_ok


def module_for(mv, E, mode=None):
    vq = mv.VectorQuantizer(E.shape[0], E.shape[1]).cuda()
    with torch.no_grad():
        vq.embedding.weight.copy_(E)
    if mode is not None:
        vq.search_mode = mode
    return vq


# ------------------------------------------------------------------------------------------- golden
@pytest.mark.parametrize("mode", [0, 1, 2], ids=["auto", "exact", "tensor"])
@pytest.mark.parametrize("tag", TAGS)
def test_forward_backward_match_reference_golden(mv, ov, tag, mode):
    z = torch.from_numpy(GOLD[f"{tag}_z"])
    E = torch.from_numpy(GOLD[f"{tag}_E"])
    r = torch.from_numpy(GOLD[f"{tag}_r"])
    vq = module_for(mv, E, mode)
    zc = z.cuda().requires_grad_(True)
    q, commit, embed, idx = vq(zc)
    assert idx.dtype == torch.int64 and idx.shape == (z.shape[0] * z.shape[2] * z.shape[3],)
    assert q.shape == z.shape and commit.dim() == 0 and embed.dim() == 0
    ties = ov.tie_rows(z, E).numpy()
    mism = idx.cpu().numpy() != GOLD[f"{tag}_idx"]
    assert not np.any(mism & ~ties), f"{int((mism & ~ties).sum())} index mismatches outside fp32-tie rows"
    if tag == "trained":
        assert not mism.any() and not ties.any(), f"{int(mism.sum())} mismatches / {int(ties.sum())} tie rows on the no-tie fixture"
    if tag == "dup":
        assert not mism.any(), "duplicated codebook rows are exact ties: the FIRST index must win like torch.argmin"
    ok, codes_ok = _agreeing(mism, idx.cpu().numpy(), GOLD[f"{tag}_idx"], E.shape[0])
    assert ok.sum() >= 0.99 * ok.size                                # ties are rare: the comparisons below cover >= 99 % of the rows
    np.testing.assert_array_equal(_rows(q.detach().cpu().numpy())[ok], _rows(GOLD[f"{tag}_q"])[ok])   # fl(z + fl(q - z)) bit for bit
    # a tie row changes (q - z)^2 by a few ulps of ONE of N*D terms: the losses hold their tolerance regardless
    np.testing.assert_allclose(float(commit), float(GOLD[f"{tag}_commit"]), rtol=1e-5)
    np.testing.assert_allclose(float(embed), float(GOLD[f"{tag}_embed"]), rtol=1e-5)
    if not mism.any():
        assert vq.last_codebook_usage_percentage() == pytest.approx(float(GOLD[f"{tag}_usage"]))
        assert vq.get_codebook_usage_percentage_from_indices(idx) == pytest.approx(float(GOLD[f"{tag}_usage"]))
    (torch.sum(q * r.cuda()) + 0.7 * commit + 1.3 * embed).backward()
    np.testing.assert_allclose(_rows(zc.grad.cpu().numpy())[ok], _rows(GOLD[f"{tag}_dz"])[ok], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(vq.embedding.weight.grad.cpu().numpy()[codes_ok], GOLD[f"{tag}_dE"][codes_ok], rtol=1e-4, atol=1e-8)


def test_duplicate_codebook_rows_pick_first_index(mv):
    z = torch.from_numpy(GOLD["dup_z"]).cuda()
    E = torch.from_numpy(GOLD["dup_E"]).cuda()
    for mode in (1, 2):
        idx = mv.code_indices(z, E, mode)
        assert int(idx.max()) < 256        # rows 256.. duplicate rows 0..255: exact ties -> first index (vq_vae.py:39)
        np.testing.assert_array_equal(idx.cpu().numpy(), GOLD["dup_idx"])


# ----------------------------------------------------------------------------- tensor path vs oracle
@pytest.mark.parametrize("codebook", ["init", "trained"])
@pytest.mark.parametrize("shape", [(128, 8, 8), (16, 64, 64), (3, 7, 9), (1, 1, 1), (2, 5, 13), (128, 1, 1), (129, 1, 1), (43, 1, 3)],
                         ids=["vqvae_cifar_b128", "N65536", "ragged_hw63", "single_row", "N130", "hw1_one_tile", "hw1_N129", "hw3_N129"])
def test_tensor_path_indices_match_oracle(mv, ov, codebook, shape):
    B, H, W = shape
    z, E = make_inputs(B, 64, H, W, 512, codebook, seed=11 + B)
    zc, Ec = z.cuda(), E.cuda()
    idx_t = mv.code_indices(zc, Ec, 2)
    n_recheck = mv.quantizer.rechecked_rows(zc.device)
    idx_e = mv.code_indices(zc, Ec, 1)
    ref = ov.code_indices(z, E).numpy()
    ties = ov.tie_rows(z, E).numpy()
    N = B * H * W
    for name, got in (("tensor", idx_t), ("exact", idx_e)):
        mism = got.cpu().numpy() != ref
        assert not np.any(mism & ~ties), f"{name}: {int((mism & ~ties).sum())} mismatches outside {int(ties.sum())} tie rows (N={N})"
    # the two CUDA paths implement the same decision rule: they must agree everywhere
    np.testing.assert_array_equal(idx_t.cpu().numpy(), idx_e.cpu().numpy())
    print(f"\n[report] {codebook} N={N}: fp32-tie rows {int(ties.sum())}, rows re-evaluated exactly by the tensor path "
          f"{n_recheck} ({100.0 * n_recheck / N:.2f}%), tensor-vs-reference mismatches {(idx_t.cpu().numpy() != ref).sum()}")


@pytest.mark.parametrize("codebook", ["init", "trained"])
def test_tensor_path_keys_are_inside_the_recheck_bound(mv, codebook):
    """The tensor core delivers sort keys  key[n, j] = score[n, j] + offset(tile)  in [M, 2M) with the column
    (bits 0, 3, 4 of j mod 32) in the 3 low mantissa bits.  The re-check threshold 1.25 M 2^-16 assumes that key differences
    reproduce exact score differences to well inside it: measure the spread of key - exact score per row."""
    z, E = make_inputs(8, 64, 16, 16, 512, codebook, seed=5)
    zc, Ec = z.cuda(), E.cuda()
    N = 8 * 16 * 16
    dbg = torch.full((N, 512), float("nan"), device="cuda")
    mv.code_indices(zc, Ec, 2, debug_scores=dbg)
    assert not torch.isnan(dbg).any()
    keys = dbg.cpu()
    bits = keys.view(torch.int32)
    cols = torch.arange(512, dtype=torch.int32)[None, :] & 31
    i3 = (cols & 1) | ((cols >> 3) << 1)                 # bits 0, 3, 4 of the column; bits 1, 2 are implied by the tracker
    assert torch.equal(bits & 7, i3.expand(N, 512)), "low mantissa bits must carry the column index"
    expo = (bits >> 23) & 0xFF
    assert (expo == expo[:, :1]).all(), "all keys of a row must share one binade"
    M = torch.ldexp(torch.ones(N, dtype=torch.float64), (expo[:, 0] - 127).to(torch.int32))
    flat = z.permute(0, 2, 3, 1).reshape(N, 64).double()
    E64 = E.double()
    exact = (E64 ** 2).sum(1)[None, :] - 2.0 * flat @ E64.t()
    delta = keys.double() - exact                      # = offset(tile) + error, per row
    spread = delta.max(dim=1).values - delta.min(dim=1).values
    rel = (spread / M).max().item()
    print(f"\n[report] {codebook}: max over rows of spread(key - exact score) / M = {rel:.3e}  (re-check threshold 1.25 * 2^-16 = {1.25 * 2 ** -16:.3e})")
    assert rel < 1.25 * 2.0 ** -16


def test_planted_codes_are_recovered_at_full_size(mv):
    """Size-independent property at the largest BASELINE shape (VQ-VAE2 bottom, N = 262,144): latents
    that ARE codebook rows (plus noise far below the inter-code spacing) decode to the planted code."""
    g = torch.Generator(device="cuda").manual_seed(3)
    K, D, B, H, W = 512, 64, 64, 64, 64
    E = 0.5 * torch.randn(K, D, generator=g, device="cuda")
    planted = torch.randint(0, K, (B * H * W,), generator=g, device="cuda")
    flat = E[planted] + 1e-3 * torch.randn(B * H * W, D, generator=g, device="cuda")
    z = flat.view(B, H, W, D).permute(0, 3, 1, 2).contiguous()
    vq = module_for(mv, E.cpu())
    q, commit, embed, idx = vq(z)
    assert torch.equal(idx, planted)
    assert float(commit) == pytest.approx(1e-6, rel=0.05) and float(commit) == float(embed)
    # idempotence: quantizing the quantized output selects the same codes
    assert torch.equal(vq.get_code_indices(q.detach()), planted)
    assert vq.last_codebook_usage_percentage() == 100.0


@pytest.mark.parametrize("codebook", ["init", "trained"])
def test_large_search_staged_recheck_matches_exact_mode(mv, codebook):
    """N > 2^19 rows: the worklist is re-evaluated by the STAGED exact kernel (smaller searches use the direct one, covered
    above against the oracle).  Size-independent check: the tensor path must agree with the all-rows exact mode, which is
    held to the oracle at the sizes the oracle finishes in seconds."""
    B, H, W = 130, 64, 64                                       # N = 532,480
    g = torch.Generator(device="cuda").manual_seed(17)
    z = 0.5 * torch.randn(B, 64, H, W, generator=g, device="cuda")
    E = (0.5 * torch.randn(512, 64, generator=g, device="cuda") if codebook == "trained"
         else (torch.rand(512, 64, generator=g, device="cuda") * 2 - 1) / 512)
    idx_t = mv.code_indices(z, E, 2)
    n_recheck = mv.quantizer.rechecked_rows(z.device)
    idx_e = mv.code_indices(z, E, 1)
    assert torch.equal(idx_t, idx_e)
    assert 0 < n_recheck < 0.02 * B * H * W


@pytest.mark.parametrize("shape", [(4, 8, 8), (40, 64, 64)], ids=["direct_recheck", "N163840"])
def test_non_finite_and_huge_latents_stay_in_range(mv, ov, shape):
    """Diverged training (the reference only warns, main.py:163-164): rows with inf / NaN / overflowing latents must not crash
    or produce out-of-range indices; every non-finite row gets torch.argmin's index (the first NaN distance, or code 0 when
    every distance overflows to inf -- decided by where the inf / NaN terms fall, not by rounding); every finite row keeps
    its exact index."""
    B, H, W = shape
    z, E = make_inputs(B, 64, H, W, 512, "trained", seed=99)
    z[0, :, 0, 0] = float("inf")
    z[0, 3, 0, 1] = float("nan")
    z[1, :, 2, 3] = 1e20                                      # |z|^2 overflows float32 -> every distance is inf
    z[2, 5, 1, 1] = -3e19
    vq = module_for(mv, E)
    q, commit, embed, idx = vq(z.cuda())
    torch.cuda.synchronize()
    idx = idx.cpu()
    assert int(idx.min()) >= 0 and int(idx.max()) < 512
    ref = ov.code_indices(z, E)
    HW = H * W
    assert int(idx[1 * HW + 2 * W + 3]) == 0 == int(ref[1 * HW + 2 * W + 3])
    finite = torch.isfinite(z).all(dim=1).reshape(-1) & (z.abs().amax(dim=1).reshape(-1) < 1e18)
    assert int((~finite).sum()) == 4 and torch.equal(idx[~finite], ref[~finite])
    ties = ov.tie_rows(torch.nan_to_num(z, nan=0.0, posinf=0.0, neginf=0.0).clamp(-10, 10), E)
    assert not bool(((idx != ref) & finite & ~ties).any())


# ------------------------------------------------------------------------------- general (K, D) path
@pytest.mark.parametrize("K,D,shape", [(100, 48, (3, 5, 7)), (512, 32, (4, 8, 8)), (37, 3, (2, 4, 4)), (1024, 64, (2, 8, 8)),
                                       (256, 64, (4, 8, 8))])
def test_exact_path_other_shapes(mv, ov, K, D, shape):
    B, H, W = shape
    z, E = make_inputs(B, D, H, W, K, "trained", seed=K + D)
    vq = module_for(mv, E)
    zc = z.cuda().requires_grad_(True)
    q, commit, embed, idx = vq(zc)
    zr = z.clone().requires_grad_(True)
    Er = E.clone().requires_grad_(True)
    q_ref, c_ref, e_ref, idx_ref = ov.quantize_forward(zr, Er)
    ties = ov.tie_rows(z, E).numpy()
    mism = idx.cpu().numpy() != idx_ref.numpy()
    assert not np.any(mism & ~ties)
    assert not mism.any(), f"{int(mism.sum())} tie-row mismatches on a trained-like codebook (expected none)"
    np.testing.assert_array_equal(q.detach().cpu().numpy(), q_ref.detach().numpy())
    np.testing.assert_allclose(float(commit), float(c_ref), rtol=1e-5)
    r = torch.randn(z.shape, generator=torch.Generator().manual_seed(1))
    (torch.sum(q * r.cuda()) + 0.7 * commit + 1.3 * embed).backward()
    (torch.sum(q_ref * r) + 0.7 * c_ref + 1.3 * e_ref).backward()
    np.testing.assert_allclose(zc.grad.cpu().numpy(), zr.grad.numpy(), rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(vq.embedding.weight.grad.cpu().numpy(), Er.grad.numpy(), rtol=1e-4, atol=1e-8)


@pytest.mark.parametrize("shape", [(5, 8, 12), (3, 4, 8), (16, 64, 64), (300, 8, 8), (3, 7, 9), (129, 1, 1), (7, 4, 5), (2, 5, 13),
                                   (40, 16, 16)],
                         ids=["hw96_tail_unit", "hw32", "N65536_multi_unit", "hw64_N19200", "ragged_hw63", "hw1_N129", "hw20", "hw65",
                              "hw256_N10240"])
def test_backward_k512_both_dE_kernels_match_oracle(mv, ov, shape):
    """K6 at K = 512, D = 64: H*W % 32 == 0 runs the tensor-map (TMA) codebook-gradient kernel, everything else the
    cp.async one; both against autograd through the reference expressions (oracle).  dz rtol 1e-5, dE rtol 1e-4
    (float32 sums of up to N rows in a different order), and bit-reproducible run to run."""
    B, H, W = shape
    z, E = make_inputs(B, 64, H, W, 512, "trained", seed=B * 1000 + H * W)
    vq = module_for(mv, E)
    zr = z.clone().requires_grad_(True)
    Er = E.clone().requires_grad_(True)
    q_ref, c_ref, e_ref, idx_ref = ov.quantize_forward(zr, Er)
    r = torch.randn(z.shape, generator=torch.Generator().manual_seed(1))
    (torch.sum(q_ref * r) + 0.7 * c_ref + 1.3 * e_ref).backward()
    grads = []
    for _ in range(2):
        zc = z.cuda().requires_grad_(True)
        vq.embedding.weight.grad = None
        q, commit, embed, idx = vq(zc)
        mism = idx.cpu().numpy() != idx_ref.numpy()
        # trained-like codebook: at most a couple of fp32-tie rows (SURVEY App. C.1: 1 row within 4 ulp at N = 65,536);
        # they are excluded row by row (and the codes they touch), nothing else is ever skipped
        assert not np.any(mism & ~ov.tie_rows(z, E).numpy()) and mism.sum() <= 2, f"{int(mism.sum())} index mismatches"
        (torch.sum(q * r.cuda()) + 0.7 * commit + 1.3 * embed).backward()
        grads.append((zc.grad.cpu().numpy(), vq.embedding.weight.grad.cpu().numpy()))
    ok, codes_ok = _agreeing(mism, idx.cpu().numpy(), idx_ref.numpy(), 512)
    np.testing.assert_allclose(_rows(grads[0][0])[ok], _rows(zr.grad.numpy())[ok], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(grads[0][1][codes_ok], Er.grad.numpy()[codes_ok], rtol=1e-4, atol=1e-8)
    np.testing.assert_array_equal(grads[0][0], grads[1][0])
    np.testing.assert_array_equal(grads[0][1], grads[1][1])


# ------------------------------------------------------------------------------------ module contract
def test_module_contract(mv):
    vq = mv.VectorQuantizer(512, 64).cuda()
    assert list(vq.state_dict().keys()) == ["embedding.weight"]                  # checkpoint key (SURVEY 5)
    assert vq.K == 512 and vq.D == 64
    w = vq.embedding.weight
    assert float(w.abs().max()) <= 1 / 512 + 1e-9 and float(w.abs().max()) > 0.9 / 512   # U(-1/K, 1/K)
    z = torch.randn(2, 64, 4, 4, device="cuda")
    vq._summary_mode = True
    out = vq(z)
    assert isinstance(out, torch.Tensor) and out.shape == z.shape                # bare tensor in summary mode (vq_vae.py:59-60)
    vq._summary_mode = False
    assert len(vq(z)) == 4
    assert vq.embed_code(torch.tensor([0, 5], device="cuda")).shape == (2, 64)
    used = vq.get_used_embeddings(z)
    assert vq.get_codebook_usage_percentage(z) == pytest.approx(100.0 * used.numel() / 512)
    # non-contiguous (channels-last style) input is accepted like the reference accepts it
    znc = torch.randn(2, 4, 4, 64, device="cuda").permute(0, 3, 1, 2)
    q1 = vq(znc)[0]
    q2 = vq(znc.contiguous())[0]
    assert torch.equal(q1, q2)
    with pytest.raises(TypeError):
        vq(z.double())
    with pytest.raises(RuntimeError):
        vq(torch.randn(2, 32, 4, 4, device="cuda"))
    with pytest.raises(RuntimeError, match="CUDA"):
        vq(z.cpu())


def test_gradients_only_where_the_reference_has_them(mv):
    """commitment_loss -> latents only; embedding_loss -> codebook only; quantized -> latents only (STE)."""
    vq = mv.VectorQuantizer(512, 64).cuda()
    z = torch.randn(2, 64, 8, 8, device="cuda", requires_grad=True)
    q, commit, embed, _ = vq(z)
    gz, gE = torch.autograd.grad(commit, [z, vq.embedding.weight], retain_graph=True, allow_unused=True)
    assert gz is not None and float(gz.abs().sum()) > 0 and gE is None
    gz, gE = torch.autograd.grad(embed, [z, vq.embedding.weight], retain_graph=True, allow_unused=True)
    assert gz is None and float(gE.abs().sum()) > 0          # None, not zeros: mtl_backward skips the row's backward pass
    gz, gE = torch.autograd.grad(q.sum(), [z, vq.embedding.weight], allow_unused=True)
    assert torch.equal(gz, torch.ones_like(z)) and gE is None


def test_tensor_path_is_one_launch_and_equals_the_exact_kernel_at_scale(mv):
    """K4 re-checks its undecidable rows itself (shared-memory ring served by the producer warps): tensor mode == exact
    mode row for row on a ragged, multi-tile-per-CTA shape and on the init codebook (many near ties), the re-check count
    is reported per search, and a second search does not inherit it."""
    g = torch.Generator(device="cuda").manual_seed(7)
    z = 0.5 * torch.randn(37, 64, 24, 20, generator=g, device="cuda")       # 17,760 rows: odd number of tiles, ragged tail
    for E in (0.5 * torch.randn(512, 64, generator=g, device="cuda"),
              (torch.rand(512, 64, generator=g, device="cuda") * 2 - 1) / 512):
        idx = mv.code_indices(z, E, 2)
        n1 = mv.quantizer.rechecked_rows(z.device)
        ref = mv.code_indices(z, E, 1)
        assert int((idx != ref).sum()) == 0
        assert 0 < n1 < z.shape[0] * z.shape[2] * z.shape[3] // 20
        mv.code_indices(z[:1], E, 2)
        assert mv.quantizer.rechecked_rows(z.device) <= 480
    zbig = 0.5 * torch.randn(64, 64, 128, 128, generator=g, device="cuda")  # 1,048,576 rows: ~55 tiles per CTA
    E = 0.5 * torch.randn(512, 64, generator=g, device="cuda")
    assert int((mv.code_indices(zbig, E, 2) != mv.code_indices(zbig, E, 1)).sum()) == 0


def test_every_row_undecidable_still_terminates_and_is_exact(mv):
    """A codebook of 512 identical rows makes EVERY row undecidable on the tensor path: the re-check ring fills up and the
    epilogue has to wait for the producer warps (back-pressure, no deadlock); every row must come out as code 0."""
    g = torch.Generator(device="cuda").manual_seed(11)
    z = 0.5 * torch.randn(16, 64, 32, 32, generator=g, device="cuda")       # 16,384 rows, 128 tiles
    E = (0.5 * torch.randn(1, 64, generator=g, device="cuda")).repeat(512, 1).contiguous()
    idx = mv.code_indices(z, E, 2)
    torch.cuda.synchronize()
    assert int(idx.abs().sum()) == 0
    assert mv.quantizer.rechecked_rows(z.device) == 16 * 32 * 32
