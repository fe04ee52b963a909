"""The quantizer kernels after the search (K5 gather + losses + usage, K6a dz, K6b + its reduce dE, the EMA codebook
update) at the sizes VQ-VAE-2 and the benchmark run, where their grid-stride loops and shared-memory rings turn over.

Method: exact-grid data with planted indices.  z, the codebook E, the upstream gradients and the EMA state are drawn
from dyadic grids (z and E: m / 16 with integer |m| <= 32), and the index tensor is chosen by the test, not by the
search, so that it can be steered at what stresses K6b's routing: hot codes, owner-range boundaries, long runs.  On this
data every float32 partial sum the kernels form is exact (a CTA's partial stays below 2^20 with steps of 1/16), so the
float64 references below equal the kernels' results in any summation order and the checks are bit for bit:

    counts          torch.bincount
    S_j             float64 index_add of the rows, rounded once to float32 (EMA statistics)
    dE              (float)(ce * (count_j e_j - S_j)) in float64, ce = (double)g_embed * (double)(2.0f / (float)(N D)),
                    added in float32 into whatever dE held
    quantized       torch's float32 z + (E[idx] - z) (correctly rounded; also with Gaussian z)
    losses          float64 sum of fl32(q - z)^2 / (N D)  (Gaussian z: within the error of per-row float32 chains)
    dz              the float64 value of fmaf(cc, z - q, go): bit for bit where it is exact (no go, or grid data with
                    N D a power of two; dz64_is_exact), within one float32 ulp elsewhere
    EMA             tests/oracle_vq_ema.py with decay 0.5: cluster_size and embed_avg exact, the codebook within one ulp

The CPU tests at the top check that these references are what they claim to be and that every shape below really lands
on the kernel variant it names, with its ring turning over; they need no GPU.  The launch rules they restate are those
of launch_k6b_partials / launch_vq_backward (csrc/vq_backward.cu) and launch_vq_gather (csrc/vq_gather.cu).
"""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

import oracle_vq_ema as oe

# ---------------------------------------------------------------------------------------------- launch rules
SMS = 148                        # B200
K6B_ROWS, K6B_MAX_GRID = 128, 160
TM_DEPTH, TM_CONSUMERS = 6, 28   # tensor-map K6b: ring depth, owner warps (31 - 3 routers)
BW_DEPTH = 3                     # cp.async K6b: ring depth
SMALL_N, STREAM_THREADS = 32768, 512     # K5 / K6a: unstaged at or below SMALL_N, else min(N / 512, SMs) CTAs, grid-stride


def tm_owner(code):
    return (code * TM_CONSUMERS) >> 9


def tm_first(w):
    return (w * 512 + TM_CONSUMERS - 1) // TM_CONSUMERS


def k6b_variant(HW, z_offset=0, idx_offset=0):
    return "tma" if HW % 32 == 0 and z_offset % 16 == 0 and idx_offset % 16 == 0 else "cp_async"


def k6b_grid(N, sms=SMS):
    return min(-(-N // K6B_ROWS), K6B_MAX_GRID, sms)


def k6b_units_per_cta(N, sms=SMS):
    """Most 128-row units (tiles) any CTA of K6b processes."""
    return -(-(-(-N // K6B_ROWS)) // k6b_grid(N, sms))


def stream_passes(N, sms=SMS):
    """Most grid-stride passes any CTA of the staged K5 / K6a makes."""
    blocks = -(-N // STREAM_THREADS)
    return -(-blocks // min(blocks, sms))


# ---------------------------------------------------------------------------------------------- cases
# (B, H, W, z byte offset, idx byte offset); K = 512, D = 64
K6B_CASES = {
    "tma_N262144": (64, 64, 64, 0, 0),              # VQ-VAE-2 bottom level, ~14 units per CTA
    "tma_N4194304": (256, 128, 128, 0, 0),          # the benchmark shape, ~222 units per CTA
    "tma_N262176_tail32": (2731, 8, 12, 0, 0),      # H W = 96: the last unit has 32 rows
    "cp_hw63": (4200, 7, 9, 0, 0),                  # ~14 tiles per CTA
    "cp_hw1_ragged": (300001, 1, 1, 0, 0),          # the last tile has 97 rows
    "cp_z_misaligned": (64, 64, 64, 4, 0),          # a tensor-map shape pushed onto the fallback by z's address
    "cp_idx_misaligned": (64, 64, 64, 0, 8),        # ... and by idx's address
}
STREAM_CASES = {k: K6B_CASES[k] for k in ("tma_N262144", "tma_N4194304", "tma_N262176_tail32", "cp_hw63", "cp_hw1_ragged")}

OWNER = 13
BOUNDARY_CODES = sorted({c for w in range(1, TM_CONSUMERS) for c in (tm_first(w) - 1, tm_first(w))})


def make_idx(dist, N, g=None, device="cpu"):
    """int64 [N] code indices of one of the distributions that stress K6b's routing."""
    n = torch.arange(N, device=device)
    if dist == "uniform":
        return torch.randint(0, 512, (N,), generator=g, device=device)
    if dist == "all_code0":
        return torch.zeros(N, dtype=torch.int64, device=device)
    if dist == "all_code511":
        return torch.full((N,), 511, dtype=torch.int64, device=device)
    if dist == "one_owner":                         # every row to one owner warp's 18-19 codes
        lo, hi = tm_first(OWNER), tm_first(OWNER + 1)
        return torch.randint(lo, hi, (N,), generator=g, device=device)
    if dist == "owner_boundaries":                  # only the codes on either side of each owner boundary
        codes = torch.tensor(BOUNDARY_CODES, device=device)
        return codes[torch.randint(0, len(BOUNDARY_CODES), (N,), generator=g, device=device)]
    if dist == "one_code_per_unit":
        return (n // K6B_ROWS) % 512
    if dist == "sorted_runs":
        return n * 512 // N
    if dist == "distinct_per_unit":                 # every 128-row unit hits 128 distinct codes, spread over all owners
        return (n % K6B_ROWS) * 4 + (n // K6B_ROWS) % 4
    raise ValueError(dist)


DISTS = ("uniform", "all_code0", "all_code511", "one_owner", "owner_boundaries", "one_code_per_unit", "sorted_runs",
         "distinct_per_unit")


def grid_tensor(shape, g, device, lim=32, step=16.0):
    """float32 values m / step, integer |m| <= lim."""
    return torch.randint(-lim, lim + 1, shape, generator=g, device=device, dtype=torch.float32).div_(step)


# ---------------------------------------------------------------------------------------------- references
def rows_nchw(z, b0, b1):
    return z[b0:b1].permute(0, 2, 3, 1).reshape(-1, z.shape[1])


def chunks(z, rows=1 << 21):
    """(b0, b1) image ranges of about `rows` code vectors: the float64 references of N = 4.2 M are built in pieces."""
    B, _, H, W = z.shape
    step = max(1, rows // (H * W))
    return [(b0, min(B, b0 + step)) for b0 in range(0, B, step)]


def ref_stats(z, idx, K):
    """(count [K] int64, S [K, D] float64): exact on grid data in any summation order."""
    HW = z.shape[2] * z.shape[3]
    S = torch.zeros(K, z.shape[1], dtype=torch.float64, device=z.device)
    for b0, b1 in chunks(z):
        S.index_add_(0, idx[b0 * HW:b1 * HW], rows_nchw(z, b0, b1).double())
    return torch.bincount(idx, minlength=K), S


def f32_scale(N, D):
    """2.0f / (float)(N D), as the kernels form it."""
    return np.float32(2.0) / np.float32(float(N) * float(D))


def ref_dE(count, S, E, g_embed, N, into=None):
    """into + (float)(ce (count_j e_j - S_j)) with the bracket in float64 and a float32 add, the formula of
    vq_dE_reduce_kernel (into None: zeros, so that an empty code gives +0)."""
    ce = float(np.float64(np.float32(g_embed)) * np.float64(f32_scale(N, E.shape[1])))
    base = torch.zeros_like(E) if into is None else into
    return base + (ce * (count.double()[:, None] * E.double() - S)).float()


def ref_forward(z, E, idx):
    """(quantized [B, D, H, W] float32 = z + (E[idx] - z), sum over rows of fl32(q - z)^2 in float64)."""
    HW = z.shape[2] * z.shape[3]
    q = torch.empty_like(z)
    t = 0.0
    for b0, b1 in chunks(z):
        zc = z[b0:b1]
        e = E[idx[b0 * HW:b1 * HW]].view(b1 - b0, z.shape[2], z.shape[3], -1).permute(0, 3, 1, 2)
        diff = e - zc
        q[b0:b1] = zc + diff
        t += float((diff.double() ** 2).sum())
    return q, t


def ref_dz64(z, E, idx, go, g_commit, N):
    """float64 value of fmaf(cc, z - q, go) with cc = fl32(g_commit) * fl32(2 / (N D)) as K6a forms it, for the images
    of z (idx: their rows; N: the rows of the whole batch); go None = 0."""
    B, D, H, W = z.shape
    cc = float(np.float32(g_commit) * f32_scale(N, D))
    e = E[idx].view(B, H, W, D).permute(0, 3, 1, 2)
    v = cc * (z - e).double()
    return v if go is None else v + go.double()


def dz64_is_exact(N, D, grid, with_go):
    """Whether ref_dz64 is exact, so that its float32 rounding is fmaf's result bit for bit: cc (z - q) always is (24-bit
    cc, 24-bit difference); adding a grid go keeps it exact when z is on the grid and N D is a power of two (cc has one
    significant bit per bit of g_commit).  Checked by test_dz_reference_is_exact_on_the_grid."""
    return not with_go or (grid and (N * D) & (N * D - 1) == 0)


def ulp32(x):
    """float32 ulp of |x| (float64 tensor in, float64 out)."""
    a = x.abs().float().clamp(min=torch.finfo(torch.float32).tiny)
    return (torch.nextafter(a, torch.full_like(a, float("inf"))) - a).double()


def within_one_ulp(got, want64):
    return bool(((got.double() - want64).abs() <= ulp32(want64)).all())


def bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# ============================================================================================ CPU: the references
def test_grid_sums_are_order_independent():
    """float32 sums of grid values in any order equal the float64 sum, up to the largest partial any kernel forms: one
    K6b CTA that receives every row of its 222 units at N = 4.2 M (S stays below 2^20, at steps of 1/16)."""
    rng = np.random.default_rng(0)
    rows = k6b_units_per_cta(256 * 128 * 128) * K6B_ROWS
    assert rows * 2 < 2 ** 20
    for vals in (rng.integers(-32, 33, rows) / 16.0, np.full(rows, 2.0), np.full(rows, -2.0),
                 np.concatenate([np.full(rows // 2, 2.0), rng.integers(-32, 33, rows - rows // 2) / 16.0])):
        want = vals.sum(dtype=np.float64)
        for _ in range(3):
            perm = vals[rng.permutation(rows)].astype(np.float32)
            assert np.cumsum(perm, dtype=np.float32)[-1] == want          # sequential float32 chain
            assert perm.sum(dtype=np.float32) == want                     # numpy's pairwise order
    # the per-row loss chain of K5: 64 squares of (q - z), |q - z| <= 4 at steps of 1/16
    d = rng.integers(-64, 65, (1000, 64)) / 16.0
    d[0] = 4.0
    acc = np.zeros(1000, dtype=np.float32)
    for k in range(64):
        acc = (acc.astype(np.float64) + (d[:, k] ** 2)).astype(np.float32)
    np.testing.assert_array_equal(acc, (d ** 2).sum(1))


def test_dz_reference_is_exact_on_the_grid():
    """Where dz64_is_exact says so, the float64 value of fmaf(cc, z - q, go) is exact, so its float32 rounding is the
    fmaf result bit for bit; elsewhere it is not always exact (the GPU tests then allow one ulp).  Checked with rational
    arithmetic on the extremes and on random points, grid and Gaussian."""
    rng = np.random.default_rng(1)
    for B, H, W, _, _ in list(K6B_CASES.values()) + [(64, 64, 64, 0, 0)]:
        N = B * H * W
        for g_commit in (0.75, 0.25):
            cc = float(np.float32(g_commit) * f32_scale(N, 64))
            go = list(rng.integers(-32, 33, 300) / 16.0) + [2.0, -2.0, 1 / 16, -1 / 16, 0.0] * 2
            grid_d = list(rng.integers(-64, 65, 300) / 16.0) + [4.0, -4.0, 1 / 16, -1 / 16, 0.0, 0.0625, -0.0625, 4.0, 2.0, 1.0]
            gauss_d = [float(np.float32(v)) for v in rng.normal(0, 1, 310)]     # fl32(z - q) of Gaussian latents
            for grid, diffs in ((True, grid_d), (False, gauss_d)):
                for with_go in (False, True):
                    exact = all(Fraction(cc * a + (b if with_go else 0.0)) == Fraction(cc) * Fraction(a) + Fraction(b if with_go else 0.0)
                                for a, b in zip(diffs, go))
                    if dz64_is_exact(N, 64, grid, with_go):
                        assert exact, (N, g_commit, grid, with_go)


def test_exact_references_agree_with_the_oracle():
    """The replicated dE, dz, quantized and loss formulas equal oracle/vq.py's quantize_forward / quantize_backward on a
    small grid case (N D and the upstream gradients powers of two, indices from the oracle's own search)."""
    from oracle import vq as ov

    g = torch.Generator().manual_seed(5)
    B, D, H, W, K = 2, 64, 4, 4, 512                 # N D = 2048: float32 mse_loss of the oracle is exact too
    z = grid_tensor((B, D, H, W), g, "cpu")
    E = grid_tensor((K, D), g, "cpu")
    q_o, commit_o, embed_o, idx = ov.quantize_forward(z, E)
    N = B * H * W
    q, t = ref_forward(z, E, idx)
    assert bits_equal(q, q_o)
    loss = np.float32(t / (N * D))
    assert loss == np.float32(commit_o.item()) == np.float32(embed_o.item())
    go = grid_tensor(z.shape, g, "cpu")
    dz_o, dE_o = ov.quantize_backward(z, E, idx, go, 0.25, 0.5)
    assert bits_equal(ref_dz64(z, E, idx, go, 0.25, N).float(), dz_o) and dz64_is_exact(N, D, True, True)
    count, S = ref_stats(z, idx, K)
    assert bits_equal(ref_dE(count, S, E, 0.5, N), dE_o)
    assert int(count.sum()) == N and not bool((S != S.float().double()).any())


def test_ema_reference_matches_the_float64_oracle_on_grid_data():
    """cluster_size and embed_avg of oracle_vq_ema.ema_update_fp64 with decay 0.5 on grid data are float32 values:
    the kernels' float32 stores of them are exact."""
    g = torch.Generator().manual_seed(6)
    z = grid_tensor((4, 64, 8, 8), g, "cpu")
    idx = make_idx("uniform", 256, g)
    cs0 = torch.randint(0, 41, (512,), generator=g).float()
    ea0 = grid_tensor((512, 64), g, "cpu")
    cs, ea, _ = oe.ema_update_fp64(oe.rows(z), idx, cs0, ea0, 0.5, 1e-5)
    assert torch.equal(cs.float().double(), cs) and torch.equal(ea.float().double(), ea)


@pytest.mark.parametrize("case", sorted(K6B_CASES))
def test_cases_land_on_the_intended_kernel_variant_and_turn_their_rings(case):
    B, H, W, zo, io = K6B_CASES[case]
    N, HW = B * H * W, H * W
    variant = k6b_variant(HW, zo, io)
    assert variant == {"tma": "tma", "cp": "cp_async"}[case.split("_")[0]]
    units = k6b_units_per_cta(N)
    if variant == "tma":
        assert units > TM_DEPTH             # a ring buffer is reused: its mbarriers enter their second phase
        assert N % 32 == 0
    else:
        assert units > BW_DEPTH
    if case == "tma_N262176_tail32":
        assert N % K6B_ROWS == 32
    if case == "cp_hw1_ragged":
        assert N % K6B_ROWS == 97
    if case in STREAM_CASES:
        assert N > SMALL_N and stream_passes(N) > 1      # staged K5 / K6a, more than one grid-stride pass


def test_index_distributions_hit_what_they_name():
    N = 262144
    own = make_idx("one_owner", N, torch.Generator().manual_seed(0))
    assert set(tm_owner(int(c)) for c in own.unique()) == {OWNER}
    bnd = make_idx("owner_boundaries", N, torch.Generator().manual_seed(0))
    assert set(int(c) for c in bnd.unique()) == set(BOUNDARY_CODES)
    assert all(tm_owner(tm_first(w)) == w and tm_owner(tm_first(w) - 1) == w - 1 for w in range(1, TM_CONSUMERS))
    per_unit = make_idx("distinct_per_unit", N).view(-1, K6B_ROWS)
    assert all(len(set(r.tolist())) == K6B_ROWS for r in per_unit[:8])
    assert int(make_idx("sorted_runs", N).max()) == 511


# ============================================================================================ GPU
@pytest.fixture(scope="module")
def mv():
    import movae_b200
    return movae_b200


@pytest.fixture(scope="module")
def L():
    from movae_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def data():
    """get(case, kind): latents [B, 64, H, W] of a case at its byte offset, on the grid or Gaussian; the last one is
    kept for the next test of the same case."""
    cache = {}

    def get(case, kind="grid"):
        key = (case, kind)
        if key not in cache:
            B, H, W, zo, _ = K6B_CASES[case]
            g = torch.Generator(device="cuda").manual_seed(B + H * W)
            buf = torch.empty(B * 64 * H * W + 4, device="cuda")
            z = buf[zo // 4:zo // 4 + B * 64 * H * W].view(B, 64, H, W)
            if kind == "grid":
                z.copy_(grid_tensor(z.shape, g, "cuda"))
            else:
                z.normal_(0.0, 0.5, generator=g)
            assert z.data_ptr() % 16 == zo
            cache.clear()                                    # one case at a time: N = 4.2 M latents are 1 GB
            cache[key] = z
        return cache[key]

    return get


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ws(nbytes):
    return torch.zeros(max(int(nbytes), 16), dtype=torch.uint8, device="cuda")


def scalar(v):
    return torch.tensor([v], dtype=torch.float32, device="cuda")


def place_idx(idx, offset):
    """idx at `offset` bytes past a 16-byte boundary."""
    buf = torch.empty(idx.numel() + 2, dtype=torch.int64, device="cuda")
    out = buf[offset // 8:offset // 8 + idx.numel()]
    out.copy_(idx)
    assert out.data_ptr() % 16 == offset
    return out


def run_backward(L, z, E, idx, go=None, g_commit=None, g_embed=None, dz=None, dE=None):
    B, D, H, W = z.shape
    K = E.shape[0]
    need = L.lib().movae_vq_backward_workspace_bytes(B * H * W, K, D)
    ws = _ws(need)
    L.check(L.lib().movae_vq_backward_f32(L.ptr(go), L.ptr(g_commit), L.ptr(g_embed), L.ptr(z), B, D, H * W, L.ptr(E), K,
                                          L.ptr(idx), L.ptr(dz), L.ptr(dE), L.ptr(ws), ws.numel(), _stream()), "vq_backward_f32")


def run_gather(L, z, E, idx):
    B, D, H, W = z.shape
    K = E.shape[0]
    q = torch.empty_like(z)
    losses = torch.empty(2, device="cuda")
    usage = torch.zeros(1, dtype=torch.int32, device="cuda")
    ws = _ws(L.lib().movae_vq_workspace_bytes(B * H * W, K, D))
    L.check(L.lib().movae_vq_gather_f32(L.ptr(z), B, D, H * W, L.ptr(E), K, L.ptr(idx), L.ptr(q), L.ptr(losses), L.ptr(usage),
                                        L.ptr(ws), ws.numel(), _stream()), "vq_gather_f32")
    return q, losses, usage


class EmaState:
    """E, cluster_size, embed_avg, E_prev on the device, 16-byte aligned."""

    def __init__(self, E, cs, ea):
        self.E, self.cs, self.ea = E.clone(), cs.clone(), ea.clone()
        self.prev = torch.full_like(E, float("nan"))

    def tensors(self):
        return self.E, self.cs, self.ea, self.prev


def ema_update(L, st, z, idx, decay, eps):
    B, D, H, W = z.shape
    K = st.E.shape[0]
    ws = _ws(L.lib().movae_vq_ema_workspace_bytes(B * H * W, K, D))
    L.check(L.lib().movae_vq_ema_update_f32(L.ptr(z), B, D, H * W, L.ptr(idx), K, decay, eps, *map(L.ptr, st.tensors()),
                                            L.ptr(ws), ws.numel(), _stream()), "vq_ema_update_f32")


def ema_split(L, st, z, idx, decay, eps):
    """Statistics, then the update from them (the data-parallel path); returns the float32 statistics."""
    B, D, H, W = z.shape
    K = st.E.shape[0]
    ws = _ws(L.lib().movae_vq_ema_workspace_bytes(B * H * W, K, D))
    stats = torch.full((K + K * D,), float("nan"), device="cuda")
    L.check(L.lib().movae_vq_ema_stats_f32(L.ptr(z), B, D, H * W, L.ptr(idx), K, L.ptr(stats), L.ptr(ws), ws.numel(), _stream()),
            "vq_ema_stats_f32")
    snapshot = stats.clone()
    L.check(L.lib().movae_vq_ema_apply_f32(L.ptr(stats), K, D, decay, eps, *map(L.ptr, st.tensors()), L.ptr(ws), ws.numel(),
                                           _stream()), "vq_ema_apply_f32")
    return snapshot


def ema_state(K, D, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    E = grid_tensor((K, D), g, "cuda")
    cs = torch.randint(0, 41, (K,), generator=g, device="cuda", dtype=torch.float32)
    ea = grid_tensor((K, D), g, "cuda")
    return E, cs, ea


def check_ema_against_oracle(st, E0, cs0, ea0, count, S, decay, eps):
    """cluster_size and embed_avg exact; the codebook within one float32 ulp of the float64 oracle; E_prev = E0."""
    cs, ea, E64 = oe.ema_update_from_stats(count, S, cs0, ea0, decay, eps)
    assert bits_equal(st.cs, cs.float()), "cluster_size"
    assert bits_equal(st.ea, ea.float()), "embed_avg"
    assert within_one_ulp(st.E, E64), f"codebook: worst error {float(((st.E.double() - E64).abs() / ulp32(E64)).max()):.3g} ulp"
    assert bits_equal(st.prev, E0), "E_prev"


# ------------------------------------------------------------------------------------------- K6b, K = 512, D = 64
@pytest.mark.gpu
@pytest.mark.parametrize("dist", DISTS)
@pytest.mark.parametrize("case", list(K6B_CASES))
def test_k6b_codebook_gradient_and_ema_statistics_are_exact(mv, L, data, case, dist):
    """dE from zero and accumulated into a non-zero dE, the EMA statistics, the fused EMA update and the split path, all
    from K6b's per-CTA partials, bit for bit against the exact references."""
    B, H, W, zo, io = K6B_CASES[case]
    N, K, D = B * H * W, 512, 64
    assert k6b_units_per_cta(N, torch.cuda.get_device_properties(0).multi_processor_count) > (
        TM_DEPTH if k6b_variant(H * W, zo, io) == "tma" else BW_DEPTH), "the ring does not turn on this device"
    z = data(case)
    g = torch.Generator(device="cuda").manual_seed(N + DISTS.index(dist))
    idx = place_idx(make_idx(dist, N, g, "cuda"), io)
    E0, cs0, ea0 = ema_state(K, D, 7)
    count, S = ref_stats(z, idx, K)

    g_embed = 1.25
    want = ref_dE(count, S, E0, g_embed, N)
    dE = torch.zeros_like(E0)
    run_backward(L, z, E0, idx, g_embed=scalar(g_embed), dE=dE)
    assert bits_equal(dE, want), f"dE: {int((dE != want).sum())} elements differ"
    dE_acc = grid_tensor((K, D), g, "cuda")
    want_acc = ref_dE(count, S, E0, g_embed, N, into=dE_acc)
    run_backward(L, z, E0, idx, g_embed=scalar(g_embed), dE=dE_acc)
    assert bits_equal(dE_acc, want_acc), "dE accumulated into a non-zero dE"

    decay, eps = 0.5, 1e-5
    split = EmaState(E0, cs0, ea0)
    stats = ema_split(L, split, z, idx, decay, eps)
    assert bits_equal(stats[:K], count.float()), "EMA statistics: counts"
    assert bits_equal(stats[K:].view(K, D), S.float()), "EMA statistics: S"
    fused = EmaState(E0, cs0, ea0)
    ema_update(L, fused, z, idx, decay, eps)
    check_ema_against_oracle(fused, E0, cs0, ea0, count, S, decay, eps)
    assert torch.equal(S.float().double(), S), "S is not float32-exact: the split path rounds it, the fused one does not"
    for a, b, name in zip(fused.tensors(), split.tensors(), ("E", "cluster_size", "embed_avg", "E_prev")):
        assert bits_equal(a, b), f"split path != fused update: {name}"


# ------------------------------------------------------------------------------------------- K5 and K6a
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["grid", "gauss"])
@pytest.mark.parametrize("case", list(STREAM_CASES))
def test_gather_losses_usage_and_dz_at_scale(mv, L, data, case, kind):
    """Staged K5 and K6a over several grid-stride passes: the quantized output bit for bit (grid and Gaussian latents),
    the losses bit for bit on the grid and within the error of per-row float32 chains otherwise, the usage count, and dz
    with and without an upstream gradient of the quantized output."""
    B, H, W, _, _ = K6B_CASES[case]
    N, K, D = B * H * W, 512, 64
    assert stream_passes(N, torch.cuda.get_device_properties(0).multi_processor_count) > 1
    z = data(case, kind)
    g = torch.Generator(device="cuda").manual_seed(N + 1)
    E = grid_tensor((K, D), g, "cuda")
    idx = make_idx("uniform" if kind == "grid" else "owner_boundaries", N, g, "cuda")

    q, losses, usage = run_gather(L, z, E, idx)
    q_ref, t = ref_forward(z, E, idx)
    assert bits_equal(q, q_ref), f"quantized: {int((q != q_ref).sum())} elements differ"
    del q, q_ref
    loss_ref = t / (N * D)
    l0, l1 = (float(v) for v in losses.cpu())
    assert l0 == l1
    if kind == "grid":
        assert l0 == float(np.float32(loss_ref))
    else:
        # per row a float32 chain of 64 fma terms (relative error <= 64 u), then float64, then one float32 rounding
        assert abs(l0 - loss_ref) <= 66 * 2.0 ** -24 * loss_ref
    assert int(usage) == int(torch.unique(idx).numel())

    g_commit = 0.75
    go = grid_tensor(z.shape, g, "cuda")
    dz = torch.empty_like(z)
    for grad_out in (None, go):
        run_backward(L, z, E, idx, go=grad_out, g_commit=scalar(g_commit), dz=dz)
        exact = dz64_is_exact(N, D, kind == "grid", grad_out is not None)
        for b0, b1 in chunks(z):
            w64 = ref_dz64(z[b0:b1], E, idx[b0 * H * W:b1 * H * W], None if grad_out is None else grad_out[b0:b1], g_commit, N)
            what = f"dz (grad_out {'NULL' if grad_out is None else 'set'}), images {b0}..{b1}"
            if exact:
                assert bits_equal(dz[b0:b1], w64.float()), f"{what}: {int((dz[b0:b1] != w64.float()).sum())} elements differ"
            else:
                assert within_one_ulp(dz[b0:b1], w64), f"{what}: more than one ulp from the float64 value"


# ------------------------------------------------------------------------------------------- other (K, D)
@pytest.mark.gpu
def test_k1024_unstaged_gather_atomic_backward_and_ema(mv, L):
    """K = 1024, D = 64 at N = 262,144: the unstaged K5 (the codebook does not fit the staging buffer), the atomic K6 and
    the atomic EMA statistics.  The atomic dE adds fl32(ce (q - z)) per row in any order: it is held to the float32
    error bound of that sum, everything else bit for bit."""
    B, H, W, K, D = 64, 64, 64, 1024, 64
    N = B * H * W
    g = torch.Generator(device="cuda").manual_seed(1024)
    z = grid_tensor((B, D, H, W), g, "cuda")
    E0, cs0, ea0 = ema_state(K, D, 8)
    idx = torch.randint(0, K, (N,), generator=g, device="cuda")

    q, losses, usage = run_gather(L, z, E0, idx)
    q_ref, t = ref_forward(z, E0, idx)
    assert bits_equal(q, q_ref)
    assert float(losses[0]) == float(losses[1]) == float(np.float32(t / (N * D)))
    assert int(usage) == int(torch.unique(idx).numel())

    go = grid_tensor(z.shape, g, "cuda")
    dz = torch.empty_like(z)
    dE = torch.zeros_like(E0)
    run_backward(L, z, E0, idx, go=go, g_commit=scalar(0.75), g_embed=scalar(1.25), dz=dz, dE=dE)
    assert dz64_is_exact(N, D, True, True) and bits_equal(dz, ref_dz64(z, E0, idx, go, 0.75, N).float())
    count, S = ref_stats(z, idx, K)
    want = ref_dE(count, S, E0, 1.25, N).double()
    ce = 1.25 * float(f32_scale(N, D))
    absum = torch.zeros(K, D, dtype=torch.float64, device="cuda")        # sum over the code's rows of |ce (q - z)|
    for b0, b1 in chunks(z):
        r = idx[b0 * H * W:b1 * H * W]
        absum.index_add_(0, r, (ce * (E0[r].double() - rows_nchw(z, b0, b1).double())).abs())
    bound = (count.double()[:, None] + 1) * 2.0 ** -24 * absum + ulp32(want)
    assert bool(((dE.double() - want).abs() <= bound).all()), "atomic dE outside the float32 summation bound"

    decay, eps = 0.5, 1e-5
    split = EmaState(E0, cs0, ea0)
    stats = ema_split(L, split, z, idx, decay, eps)
    assert bits_equal(stats[:K], count.float()) and bits_equal(stats[K:].view(K, D), S.float())
    check_ema_against_oracle(split, E0, cs0, ea0, count, S, decay, eps)
    fused = EmaState(E0, cs0, ea0)
    ema_update(L, fused, z, idx, decay, eps)
    check_ema_against_oracle(fused, E0, cs0, ea0, count, S, decay, eps)


# ------------------------------------------------------------------------------------------- reproducibility
@pytest.mark.gpu
def test_k6b_dE_and_ema_update_are_bit_reproducible_at_the_benchmark_size(mv, L, data):
    """N = 4,194,304 Gaussian latents (float32 sums that DO round): two runs give the same bits."""
    case = "tma_N4194304"
    z = data(case, "gauss")
    B, H, W, _, _ = K6B_CASES[case]
    N, K, D = B * H * W, 512, 64
    idx = torch.randint(0, K, (N,), generator=torch.Generator(device="cuda").manual_seed(4), device="cuda")
    E0, cs0, ea0 = ema_state(K, D, 9)
    runs = []
    for _ in range(2):
        dE = torch.zeros_like(E0)
        run_backward(L, z, E0, idx, g_embed=scalar(1.0), dE=dE)
        st = EmaState(E0, cs0, ea0)
        ema_update(L, st, z, idx, 0.99, 1e-5)
        runs.append((dE,) + st.tensors())
    for a, b in zip(*runs):
        assert bits_equal(a, b)
    assert float(runs[0][0].abs().max()) > 0


# ------------------------------------------------------------------------------------------- end to end
def planted_latents(g, B, H, W, K=512, D=64):
    """(z [B, D, H, W], E, planted): z = E[planted] + noise of at most 1/32 per channel, all on the 1/64 grid."""
    E = grid_tensor((K, D), g, "cuda")
    d2 = torch.cdist(E.double(), E.double()) ** 2 + torch.eye(K, device="cuda", dtype=torch.float64) * 1e9
    noise = grid_tensor((B * H * W, D), g, "cuda", lim=2, step=64.0)
    assert float(d2.min().sqrt()) > 4 * math.sqrt(D) / 32           # |noise| <= sqrt(D) / 32: the search must return `planted`
    planted = torch.randint(0, K, (B * H * W,), generator=g, device="cuda")
    z = (E[planted] + noise).view(B, H, W, D).permute(0, 3, 1, 2).contiguous()
    return z, E, planted


@pytest.mark.gpu
def test_module_forward_backward_eager_and_graph_replay_at_vqvae2_size(mv):
    """VectorQuantizer at N = 262,144 through autograd, then the same step replayed from a CUDA graph (GraphedStep, what
    the benchmark's fwd_bwd_graph_ms times): both equal the exact references bit for bit.  N D = 2^24 and the upstream
    gradients are powers of two, so oracle/vq.py's quantize_backward gives those bits."""
    from oracle import vq as ov

    B, H, W = 64, 64, 64
    N, D = B * H * W, 64
    g = torch.Generator(device="cuda").manual_seed(31)
    z, E, planted = planted_latents(g, B, H, W)
    go = grid_tensor(z.shape, g, "cuda")
    g_commit, g_embed = 0.25, 0.5
    q_ref, t = ref_forward(z, E, planted)
    loss_ref = float(np.float32(t / (N * D)))
    dz_ref, dE_ref = ov.quantize_backward(z.cpu(), E.cpu(), planted.cpu(), go.cpu(), g_commit, g_embed)
    dz_ref, dE_ref = dz_ref.cuda(), dE_ref.cuda()

    vq = mv.VectorQuantizer(512, D).cuda()
    with torch.no_grad():
        vq.embedding.weight.copy_(E)
    zg = z.clone().requires_grad_(True)
    gc, ge = torch.tensor(g_commit, device="cuda"), torch.tensor(g_embed, device="cuda")

    def step():
        q, commit, embed, idx = vq(zg)
        dz, dE = torch.autograd.grad([q, commit, embed], [zg, vq.embedding.weight], grad_outputs=[go, gc, ge])
        return q, commit, embed, idx, dz, dE

    def check(outs, what):
        q, commit, embed, idx, dz, dE = outs
        assert torch.equal(idx, planted), what
        assert bits_equal(q, q_ref), what
        assert float(commit.detach()) == float(embed.detach()) == loss_ref, what
        assert bits_equal(dz, dz_ref), f"{what}: dz"
        assert bits_equal(dE, dE_ref), f"{what}: dE"

    check(step(), "eager")
    assert vq.last_codebook_usage_percentage() == 100.0
    graphed = mv.GraphedStep(step, warmup=2)
    for _ in range(3):
        outs = graphed()
    torch.cuda.synchronize()
    check(outs, "graph replay")


@pytest.mark.gpu
def test_ema_module_training_step_at_vqvae2_size(mv):
    """One VectorQuantizerEMA training step at N = 262,144: search, gather, losses and dz from the pre-update codebook
    bit for bit, the update against the float64 oracle (cluster_size and embed_avg exact, the codebook within one ulp)."""
    from oracle import vq as ov

    B, H, W = 64, 64, 64
    N, K, D = B * H * W, 512, 64
    g = torch.Generator(device="cuda").manual_seed(37)
    z, E0, planted = planted_latents(g, B, H, W)
    cs0 = torch.randint(0, 41, (K,), generator=g, device="cuda", dtype=torch.float32)
    ea0 = grid_tensor((K, D), g, "cuda")
    go = grid_tensor(z.shape, g, "cuda")
    ema = mv.VectorQuantizerEMA(K, D, decay=0.5, epsilon=1e-5).cuda()
    with torch.no_grad():
        ema.embedding.weight.copy_(E0)
        ema.cluster_size.copy_(cs0)
        ema.embed_avg.copy_(ea0)
    zg = z.clone().requires_grad_(True)
    q, commit, embed, idx = ema(zg)
    torch.autograd.backward([q, commit], [go, torch.tensor(0.25, device="cuda")])
    assert torch.equal(idx, planted)
    q_ref, t = ref_forward(z, E0, planted)
    assert bits_equal(q.detach(), q_ref)
    assert float(commit.detach()) == float(embed.detach()) == float(np.float32(t / (N * D)))
    dz_ref, _ = ov.quantize_backward(z.cpu(), E0.cpu(), planted.cpu(), go.cpu(), 0.25, 0.0)
    assert bits_equal(zg.grad, dz_ref.cuda())
    cs, ea, E64 = oe.ema_update_fp64(oe.rows(z).cpu(), planted.cpu(), cs0.cpu(), ea0.cpu(), 0.5, 1e-5)
    assert bits_equal(ema.cluster_size.cpu(), cs.float()) and bits_equal(ema.embed_avg.cpu(), ea.float())
    assert within_one_ulp(ema.embedding.weight.detach().cpu(), E64)
    assert bits_equal(ema._pre_update, E0)
