"""Both codebook searches (K4 tcgen05 + in-kernel re-check, K4x exact kernel) against the exact model of their decision
rule (tests/oracle_vq_search.py) on EVERY row: nothing is excluded as an "fp32 tie".  The data are on grids where the
model is bit-exact (see that module), so ties are what these tests are about: planted at chosen tracker / chunk / group
positions of the tensor path's epilogue, at its decision threshold, in the regime where |z| >> |e| rounds many distances
together, at the exact kernel's variant limits, and with inf / NaN inputs (torch.argmin: the first NaN wins).

Every search writes into an index buffer pre-filled with -1, so a row a kernel never writes cannot pass by inheriting a
previous result."""
import pytest
import torch

import oracle_vq_search as os_

pytestmark = pytest.mark.gpu

EXACT, TENSOR, AUTO = 1, 2, 0
MODES = {"exact": EXACT, "tensor": TENSOR, "auto": AUTO}


@pytest.fixture(scope="module")
def L():
    from movae_b200 import _lib
    return _lib


def search(L, z, E, mode):
    """(idx int64 [N] on the device, rows the tensor path re-checked) through movae_vq_argmin_f32, the entry point of
    movae_b200.code_indices."""
    B, D, H, W = z.shape
    K = E.shape[0]
    idx = torch.full((B * H * W,), -1, dtype=torch.int64, device=z.device)
    ws = torch.zeros(max(int(L.lib().movae_vq_workspace_bytes(B * H * W, K, D)), 16), dtype=torch.uint8, device=z.device)
    L.check(L.lib().movae_vq_argmin_f32(L.ptr(z), B, D, H * W, L.ptr(E), K, L.ptr(idx), mode, L.ptr(None), L.ptr(ws), ws.numel(),
                                        torch.cuda.current_stream().cuda_stream), "vq_argmin_f32")
    torch.cuda.synchronize()
    return idx, int(ws[:4].view(torch.int32).item())


def assert_rule(L, z, E, modes, want=None):
    """idx == the model on every row, in each mode; returns {mode: rows re-checked}."""
    if want is None:
        want = os_.rule_indices(z.cpu(), E.cpu())
    rechecked = {}
    for name in modes:
        idx, n = search(L, z, E, MODES[name])
        bad = (idx.cpu() != want).nonzero().flatten()
        assert bad.numel() == 0, (f"{name}: {bad.numel()} of {want.numel()} rows differ from the rule, first rows "
                                  f"{bad[:5].tolist()}: got {idx.cpu()[bad[:5]].tolist()}, want {want[bad[:5]].tolist()}")
        rechecked[name] = n
    return rechecked


# ------------------------------------------------------------------------------------------- tensor path: planted ties
@pytest.mark.parametrize("variant", os_.VARIANTS)
@pytest.mark.parametrize("structure", sorted(os_.tie_structures()))
def test_planted_tie_structures(L, structure, variant):
    """2-5 codes equidistant or a quantum apart in one tracker, across trackers, across groups, one per tracker, and exact
    ties whose winner is not the first in tracker order; every third row sits on them.  The re-check count is what the
    keys (exact on this grid) and each tile's threshold imply."""
    z, E = os_.planted_case(structure, variant)
    lo, hi = os_.expected_rechecks(os_.rows(z), E)
    n = assert_rule(L, z.cuda(), E.cuda(), ("exact", "tensor", "auto"))
    print(f"\n[report] {structure}/{variant}: rechecked {n['tensor']} of {z.shape[0] * z.shape[2] * z.shape[3]} (expected {lo}..{hi})")
    assert lo <= n["tensor"] <= hi and n["tensor"] > 0


@pytest.mark.parametrize("side", ["inside", "outside"])
@pytest.mark.parametrize("placement", ["one_tracker", "two_trackers", "two_groups"])
def test_gap_at_the_decision_threshold(L, placement, side):
    """Two codes whose score gap is one quantum inside / outside 1.25 M 2^-16, M from the tile as the producer forms it;
    every row is the same center, so every tile has the same M: all rows re-checked, or none."""
    codes = {"one_tracker": [os_.code_at(0, 2, 1, 3), os_.code_at(0, 6, 1, 0)],
             "two_trackers": [os_.code_at(1, 1, 3, 2), os_.code_at(1, 1, 0, 5)],
             "two_groups": [os_.code_at(1, 0, 2, 0), os_.code_at(0, 7, 2, 1)]}[placement]
    g = torch.Generator().manual_seed(5)
    E = os_.coarse_grid((512, 64), g)
    center = os_.coarse_grid((64,), g, lim=10)
    z2 = float((center.double() ** 2).sum())
    M, amb = os_.tile_key_scale(z2, float((E.double() ** 2).sum(1).max()))
    thr_q = os_.recheck_threshold(M) / os_.QUANTUM
    k = int(thr_q) if side == "inside" else int(thr_q) + 1
    if side == "inside" and k == thr_q:
        k -= 1
    os_.plant(E, center, codes, [0, k])
    M2, amb2 = os_.tile_key_scale(z2, float((E.double() ** 2).sum(1).max()))
    assert M2 == M and not amb and not amb2 and k >= 1
    B, H, W = 3, 37, 41                                          # 4551 rows: 36 tiles, the last one ragged
    z = os_.to_nchw(center.repeat(B * H * W, 1), B, H, W)
    n = assert_rule(L, z.cuda(), E.cuda(), ("exact", "tensor"))
    print(f"\n[report] {placement}/{side}: threshold {thr_q:.2f} quanta, gap {k}, rechecked {n['tensor']}")
    assert n["tensor"] == (B * H * W if side == "inside" else 0)


# ------------------------------------------------------------------------------------------- tensor path: scale
def test_tensor_path_at_scale_with_an_outlier_per_tile(L):
    """N = 1,046,821 (ragged: N mod 128 = 37) fine-grid rows, one row per 128-row tile scaled by 2^10: it raises its
    tile's M, so most of the tile goes through the re-check, and the outlier itself lives where |z| >> |e|."""
    B, H, W = 61, 131, 131
    N = B * H * W
    g = torch.Generator().manual_seed(8)
    E = os_.fine_grid((512, 64), g)
    flat = os_.fine_grid((N, 64), g)
    t = torch.arange(0, N, 128)
    out = t + (t // 128 * 37) % 128
    out = out[out < N]
    flat[out] *= 2.0 ** 10
    z = os_.to_nchw(flat, B, H, W)
    want = os_.rule_indices(flat, E)
    del flat
    n = assert_rule(L, z.cuda(), E.cuda(), ("tensor", "exact"), want)
    print(f"\n[report] N={N} with outliers: rechecked {n['tensor']} ({100.0 * n['tensor'] / N:.1f}%)")
    assert N // 2 < n["tensor"] < N


def test_benchmark_size_tensor_equals_exact_and_a_sample_equals_the_rule(L):
    B, H, W = 256, 128, 128                                      # N = 4,194,304
    g = torch.Generator(device="cuda").manual_seed(9)
    z = os_.fine_grid((B, 64, H, W), g, device="cuda")
    E = os_.fine_grid((512, 64), g, device="cuda")
    idx_t, n = search(L, z, E, TENSOR)
    idx_e, _ = search(L, z, E, EXACT)
    assert int((idx_t != idx_e).sum()) == 0 and int((idx_t < 0).sum()) == 0
    rows = torch.randperm(B * H * W, generator=torch.Generator().manual_seed(10))[:65536]
    sample = z.permute(0, 2, 3, 1).reshape(-1, 64)[rows.cuda()].cpu()
    assert torch.equal(idx_t.cpu()[rows], os_.rule_indices(sample, E.cpu()))
    print(f"\n[report] N=4194304: rechecked {n} ({100.0 * n / (B * H * W):.3f}%)")
    assert 0 < n < 0.02 * B * H * W


# ------------------------------------------------------------------------------------------- rounded ties
@pytest.mark.parametrize("mode", ["exact", "tensor"])
def test_first_index_wins_where_distances_round_together(L, mode):
    """|z| ~ 2^12 |e| and codes a few fine quanta apart: ulp(|z|^2) is far above the score gaps, many codes share the
    float32 distance, and the first of them must win (the candidate bounds' ulp terms)."""
    g = torch.Generator().manual_seed(12)
    e0 = os_.fine_grid((64,), g)
    E = e0 + torch.randint(-2, 3, (512, 64), generator=g).float() * os_.FINE
    B, H, W = 2, 97, 101
    flat = os_.fine_grid((B * H * W, 64), g)
    flat[::2] *= 2.0 ** 12
    z = os_.to_nchw(flat, B, H, W)
    want = os_.rule_indices(flat, E)
    d = os_.rule_distances(flat[::2][:2000], E)
    shared = (d == d.min(1, keepdim=True).values).sum(1)
    assert float(shared.float().mean()) > 4                     # the regime: several codes at the minimal float32 distance
    assert_rule(L, z.cuda(), E.cuda(), (mode,), want)


# ------------------------------------------------------------------------------------------- exact kernel variants
@pytest.mark.parametrize("case", sorted(os_.EXACT_CASES))
def test_exact_kernel_variants(L, case):
    K, D, (B, H, W), variant = os_.EXACT_CASES[case]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert os_.exact_passes(B * H * W, K, D, sms) >= 2, "the grid-stride loop does not turn on this device"
    g = torch.Generator().manual_seed(K * 7 + D)
    E = os_.fine_grid((K, D), g)
    if K >= 4:
        E[K // 2] = E[K // 4]                                    # an exact duplicate: the first index must win
    z = os_.fine_grid((B, D, H, W), g)
    assert_rule(L, z.cuda(), E.cuda(), ("exact", "auto"))


def test_misaligned_codebook_uses_scalar_staging(L):
    K, D, (B, H, W), _ = os_.MISALIGNED_CASE
    g = torch.Generator().manual_seed(13)
    buf = torch.empty(K * D + 4, device="cuda")
    E = buf[1:1 + K * D].view(K, D)
    E.copy_(os_.fine_grid((K, D), g).cuda())
    assert E.data_ptr() % 16 == 4
    z = os_.fine_grid((B, D, H, W), g).cuda()
    n = assert_rule(L, z, E, ("exact", "auto"))
    assert n["auto"] == 0                                        # auto fell back to the exact kernel
    with pytest.raises(RuntimeError):
        search(L, z, E, TENSOR)


def test_codebook_too_large_for_the_exact_kernel_is_rejected(L):
    z = torch.zeros(1, 64, 4, 4, device="cuda")
    E = torch.zeros(os_.REJECTED_K, 64, device="cuda")
    with pytest.raises(RuntimeError, match="too large"):
        search(L, z, E, EXACT)
    with pytest.raises(RuntimeError, match="too large"):
        search(L, z, E, AUTO)


# ------------------------------------------------------------------------------------------- non-finite inputs
@pytest.mark.parametrize("name", os_.NON_FINITE)
def test_non_finite_inputs_follow_torch_argmin(L, name):
    z, E = os_.non_finite_case(name)
    assert_rule(L, z.cuda(), E.cuda(), ("exact", "tensor", "auto"))
