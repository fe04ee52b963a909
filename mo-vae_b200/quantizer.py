"""Drop-in for the reference's `VectorQuantizer` (/root/reference/models/vq_vae.py:11-124) over the
CUDA kernels K4 (tcgen05 nearest-codebook search), K5 (gather + losses + straight-through output +
usage bitmap) and K6 (backward).

Same constructor, attributes (`K`, `D`, `_summary_mode`, `embedding` = nn.Embedding(K, D) initialised
U(-1/K, 1/K), parameter name `embedding.weight`), same `forward` return tuple

    (quantized[B,D,H,W], commitment_loss, embedding_loss, encoding_inds[BHW] int64)

and the same helper methods, so the reference's model shells (vq_vae.py:329, vq_vae2.py:225,231) and
state dicts work unchanged.  CUDA-only: there is no CPU fallback.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch
from torch import Tensor, nn

from . import _lib as L

_buffers: dict = {}


def _buffer(kind: str, device: torch.device, stream: int, nbytes: int, zero: bool = True) -> Tensor:
    """The device buffer of `kind` for (device, stream), replaced by a bigger one when a call needs more bytes: "vq" (the
    search / gather workspace), "ema" (the EMA update's workspace), "k6" (K6's per-CTA partials).  A workspace is
    zero-filled when it is allocated and the kernels leave it clean; the K6 scratch (`zero=False`) is written before it
    is read.  GraphedStep keeps every buffer of this cache alive for as long as a captured graph uses it."""
    key = (kind, device.index, stream)
    buf = _buffers.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = (torch.zeros if zero else torch.empty)(nbytes, dtype=torch.uint8, device=device)
        _buffers[key] = buf
    return buf


def _workspace_bytes(n_rows: int, K: int, D: int) -> int:
    need = L.lib().movae_vq_workspace_bytes(n_rows, K, D)
    if need == 0:
        raise RuntimeError(f"movae_b200: num_embeddings={K} is not supported by this CUDA build")
    return need


def _check_inputs(latents: Tensor, weight: Tensor) -> Tuple[int, int, int, int]:
    L.require_cuda(latents, "latents")
    L.require_cuda(weight, "embedding.weight")
    if latents.dim() != 4:
        raise ValueError(f"latents must be [B, D, H, W], got shape {tuple(latents.shape)}")
    if latents.dtype != torch.float32 or weight.dtype != torch.float32:
        raise TypeError("movae_b200: the quantizer computes in float32 (got "
                        f"{latents.dtype} latents / {weight.dtype} codebook)")
    B, D, H, W = latents.shape
    K, De = weight.shape
    if De != D:
        raise RuntimeError(f"latents have {D} channels but the codebook has embedding_dim={De}")
    if latents.device != weight.device:
        raise RuntimeError("latents and the codebook must be on the same CUDA device")
    return B, D, H * W, K


def code_indices(latents: Tensor, weight: Tensor, mode: int = L.VQ_AUTO, debug_scores: Optional[Tensor] = None) -> Tensor:
    """K4 only: int64 [B*H*W] nearest-code indices (vq_vae.py:28-39; the inference-mode callers
    `get_code_indices` vq_vae.py:393-423 / vq_vae2.py:290-311 use exactly this)."""
    B, D, HW, K = _check_inputs(latents, weight)
    z = latents.detach().contiguous()
    E = weight.detach().contiguous()
    idx = torch.empty(B * HW, dtype=torch.int64, device=z.device)
    stream = L.stream_of(z)
    ws = _buffer("vq", z.device, stream, _workspace_bytes(B * HW, K, D))
    with torch.cuda.device(z.device):
        L.check(L.lib().movae_vq_argmin_f32(L.ptr(z), B, D, HW, L.ptr(E), K, L.ptr(idx), int(mode), L.ptr(debug_scores),
                                            L.ptr(ws), ws.numel(), stream), "vq_argmin_f32")
    return idx


def rechecked_rows(device: torch.device) -> int:
    """Rows the last tensor-path search on the current stream re-evaluated exactly (synchronises)."""
    key = ("vq", torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream)
    ws = _buffers.get(key)
    return 0 if ws is None else int(ws[:4].view(torch.int32).item())


def codebook_usage_count(encoding_inds: Tensor, K: int) -> Tensor:
    """int32 device scalar: |unique(encoding_inds)| via a K-bit bitmap (replaces torch.unique, vq_vae.py:121)."""
    L.require_cuda(encoding_inds, "encoding_inds")
    idx = encoding_inds.detach().reshape(-1).to(torch.int64).contiguous()
    out = torch.zeros(1, dtype=torch.int32, device=idx.device)
    stream = L.stream_of(idx)
    ws = _buffer("vq", idx.device, stream, _workspace_bytes(0, K, 1))
    with torch.cuda.device(idx.device):
        L.check(L.lib().movae_vq_usage(L.ptr(idx), idx.numel(), K, L.ptr(out), L.ptr(ws), ws.numel(), stream), "vq_usage")
    return out


def _forward(latents: Tensor, E: Tensor, mode: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """K4 + K5 with the contiguous codebook E, on the current stream: (z, idx, quantized, losses [commitment, embedding],
    usage)."""
    B, D, HW, K = _check_inputs(latents, E)
    z = latents.detach().contiguous()
    N = B * HW
    if N == 0:
        raise RuntimeError("movae_b200: empty latents")
    idx = torch.empty(N, dtype=torch.int64, device=z.device)
    quantized = torch.empty_like(z)
    losses = torch.empty(2, dtype=torch.float32, device=z.device)
    usage = torch.empty(1, dtype=torch.int32, device=z.device)
    stream = L.stream_of(z)
    ws = _buffer("vq", z.device, stream, _workspace_bytes(N, K, D))
    with torch.cuda.device(z.device):
        L.check(L.lib().movae_vq_forward_f32(L.ptr(z), B, D, HW, L.ptr(E), K, L.ptr(idx), L.ptr(quantized), L.ptr(losses),
                                             L.ptr(usage), int(mode), L.ptr(ws), ws.numel(), stream), "vq_forward_f32")
    return z, idx, quantized, losses, usage


def _backward(z: Tensor, E: Tensor, idx: Tensor, g_q: Optional[Tensor], g_commit: Optional[Tensor],
              g_embed: Optional[Tensor], want_dz: bool) -> Tuple[Optional[Tensor], Optional[Tensor]]:
    """K6 on the current stream: dz when `want_dz`, dE when `g_embed` is given (None: no codebook gradient)."""
    B, D, H, W = z.shape
    K = E.shape[0]
    dz = torch.empty_like(z) if want_dz else None
    dE = torch.zeros_like(E) if g_embed is not None else None
    if dz is None and dE is None:
        return None, None
    f32 = lambda t: None if t is None else t.detach().to(torch.float32).contiguous()  # noqa: E731
    g_q, g_commit, g_embed = f32(g_q), f32(g_commit), f32(g_embed)
    stream = L.stream_of(z)
    need = L.lib().movae_vq_backward_workspace_bytes(B * H * W, K, D) if dE is not None else 0
    scratch = _buffer("k6", z.device, stream, need, zero=False) if need else None
    with torch.cuda.device(z.device):
        L.check(L.lib().movae_vq_backward_f32(L.ptr(g_q), L.ptr(g_commit), L.ptr(g_embed), L.ptr(z), B, D, H * W, L.ptr(E), K,
                                              L.ptr(idx), L.ptr(dz), L.ptr(dE), L.ptr(scratch), need, stream), "vq_backward_f32")
    return dz, dE


class _Quantize(torch.autograd.Function):
    """forward: K4 + K5; backward: K6.  Gradients (vq_vae.py:51-55): the straight-through output
    passes its gradient to the latents unchanged, commitment_loss adds 2 (z - q) / (N D) to them,
    embedding_loss sends 2 (q - z) / (N D) to the selected codebook rows; nothing flows through argmin."""

    @staticmethod
    def forward(ctx, latents: Tensor, weight: Tensor, mode: int):
        E = weight.detach().contiguous()
        z, idx, quantized, losses, usage = _forward(latents, E, mode)
        ctx.save_for_backward(z, E, idx)
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(idx, usage)
        return quantized, losses[0], losses[1], idx, usage

    @staticmethod
    def backward(ctx, g_q, g_commit, g_embed, _g_idx, _g_usage):
        z, E, idx = ctx.saved_tensors
        # no dz when nothing reaches the latents (embedding_loss alone, vq_vae.py:52): autograd then reports the latents
        # as unused instead of back-propagating zeros.  Only embedding_loss reaches the codebook (vq_vae.py:51-55).
        want_dz = ctx.needs_input_grad[0] and not (g_q is None and g_commit is None)
        dz, dE = _backward(z, E, idx, g_q, g_commit, g_embed if ctx.needs_input_grad[1] else None, want_dz)
        return dz, dE, None


class VectorQuantizer(nn.Module):
    """Vector Quantization module for VQ-VAE (same interface as the reference's, vq_vae.py:11-124)."""

    def __init__(self, num_embeddings: int, embedding_dim: int):
        super().__init__()
        self.K = num_embeddings
        self.D = embedding_dim
        self._summary_mode = False
        self.embedding = nn.Embedding(self.K, self.D)
        self.embedding.weight.data.uniform_(-1 / self.K, 1 / self.K)
        self.search_mode = L.VQ_AUTO            # MOVAE_VQ_AUTO | _EXACT | _TENSOR (include/movae_b200.h)
        self.last_usage_count: Optional[Tensor] = None   # int32 device scalar written by K5's bitmap

    def forward(self, latents: Tensor):
        quantized, commitment_loss, embedding_loss, encoding_inds, usage = self._quantize(latents)
        self.last_usage_count = usage
        if getattr(self, "_summary_mode", False):
            return quantized
        return quantized, commitment_loss, embedding_loss, encoding_inds

    def _quantize(self, latents: Tensor):
        return _Quantize.apply(latents, self.embedding.weight, self.search_mode)

    def embed_code(self, code: Tensor) -> Tensor:
        return self.embedding(code)

    def get_code_indices(self, latents: Tensor) -> Tensor:
        """int64 [B*H*W]; K4 only, no gather / losses (inference-mode code extraction)."""
        return code_indices(latents, self.embedding.weight, self.search_mode)

    def get_used_embeddings(self, latents: Tensor) -> Tensor:
        return torch.unique(self.get_code_indices(latents))

    def get_codebook_usage_percentage(self, latents: Tensor) -> float:
        return self.get_codebook_usage_percentage_from_indices(self.get_code_indices(latents))

    def get_codebook_usage_percentage_from_indices(self, encoding_inds: Tensor) -> float:
        num_used = int(codebook_usage_count(encoding_inds, self.K).item())      # python float by contract -> one D2H
        return float((num_used / self.K) * 100.0)

    def last_codebook_usage_percentage(self) -> float:
        """Usage of the most recent forward(), from the bitmap K5 already built (no extra kernel)."""
        if self.last_usage_count is None:
            raise RuntimeError("forward() has not run yet")
        return float(int(self.last_usage_count.item()) / self.K * 100.0)


class _QuantizeEMA(torch.autograd.Function):
    """forward: K4 + K5 with the current codebook, then (training) the EMA update of the codebook in place; backward: K6a
    only.  The straight-through output and commitment_loss send to the latents what `_Quantize` sends, with q from the
    PRE-update codebook, which the update copied into `vq._pre_update`.  embedding_loss keeps its value but reaches
    nothing: its gradient is dropped, so the latents get None from it and the codebook, which is not a parameter of
    gradient descent here, gets nothing at all."""

    @staticmethod
    def forward(ctx, latents: Tensor, vq: "VectorQuantizerEMA", update: bool):
        E = vq.embedding.weight.detach()
        if not E.is_contiguous():
            raise RuntimeError("movae_b200: VectorQuantizerEMA updates embedding.weight in place and needs it contiguous")
        z, idx, quantized, losses, usage = _forward(latents, E, vq.search_mode)
        if update:
            vq._update(z, idx)
            E = vq._pre_update
        ctx.save_for_backward(z, E, idx)     # the update bumped _pre_update's version: a later update makes backward raise
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(idx, usage)
        return quantized, losses[0], losses[1], idx, usage

    @staticmethod
    def backward(ctx, g_q, g_commit, _g_embed, _g_idx, _g_usage):
        z, E, idx = ctx.saved_tensors
        if not ctx.needs_input_grad[0] or (g_q is None and g_commit is None):
            return None, None, None
        dz, _ = _backward(z, E, idx, g_q, g_commit, None, True)
        return dz, None, None


class VectorQuantizerEMA(VectorQuantizer):
    """Vector quantizer whose codebook follows an exponential moving average of the latents assigned to each code
    (van den Oord et al. 2017, App. A.1; the semantics of the `Quantize` module of rosinality/vq-vae-2-pytorch).  This is
    not the reference's rule: the reference trains the codebook by gradient through embedding_loss.

    Search, gather, losses, the returned tuple `(quantized, commitment_loss, embedding_loss, encoding_inds)` (bare
    `quantized` in `_summary_mode`) and the helpers are those of `VectorQuantizer`, so a model shell takes this class by
    swapping it in.  The codebook stays `embedding.weight` [K, D], initialised U(-1/K, 1/K), with requires_grad=False.
    Persistent buffers: `cluster_size` [K] (zeros) and `embed_avg` [K, D] (a copy of the initial codebook).

    Each forward in training mode (`self.training`, also under torch.no_grad()) runs, after the search and on the
    device, with the indices searched by the pre-update codebook:

        count_j = #{n : idx_n = j},   S_j = sum_{n : idx_n = j} z_n
        cluster_size <- decay * cluster_size + (1 - decay) * count
        embed_avg    <- decay * embed_avg    + (1 - decay) * S
        n = sum_j cluster_size_j
        smoothed_j = (cluster_size_j + epsilon) / (n + K * epsilon) * n
        E_j <- embed_avg_j / smoothed_j

    The stored cluster_size is unsmoothed; the smoothing only enters the normalisation.  A code no row selects is divided
    by a tiny smoothed_j and moves far away; that is this formulation's behaviour and is kept.  eval() forwards,
    `get_code_indices` and `CodeExtractor` change no state.

    The update writes `embedding.weight` in place (flat-parameter views, CUDA graphs and load_state_dict keep working).
    The straight-through output and commitment_loss send `d_out + g_c * 2 (z - q) / (N D)` to the latents with q from the
    pre-update codebook, which the update copies into the non-persistent buffer `_pre_update`; a second training forward
    before the first one's backward makes that backward raise (autograd's saved-tensor version check).  embedding_loss
    keeps its value but sends no gradient anywhere (in `mtl_backward` its Jacobian row is the zero row).

    `stats_reducer` (None by default): a callable applied in place to the float32 [K + K*D] tensor holding count, then S,
    between the statistics pass and the update; `parallel.install_codebook_allreduce` sets it to an all_reduce so that
    batch-sharded replicas apply the same update.  Without it the update is one fused pass (two launches at K = 512,
    D = 64)."""

    def __init__(self, num_embeddings: int, embedding_dim: int, decay: float = 0.99, epsilon: float = 1e-5):
        decay, epsilon = float(decay), float(epsilon)
        if not 0.0 <= decay < 1.0:
            raise ValueError(f"decay must be in [0, 1), got {decay}")
        if not epsilon > 0.0:
            raise ValueError(f"epsilon must be > 0, got {epsilon}")
        super().__init__(num_embeddings, embedding_dim)
        self.decay = decay
        self.epsilon = epsilon
        self.embedding.weight.requires_grad_(False)
        self.register_buffer("cluster_size", torch.zeros(self.K))
        self.register_buffer("embed_avg", self.embedding.weight.detach().clone())
        self.register_buffer("_pre_update", torch.empty(self.K, self.D), persistent=False)
        self.stats_reducer: Optional[Callable[[Tensor], None]] = None
        self._stats: Optional[Tensor] = None

    def _quantize(self, latents: Tensor):
        return _QuantizeEMA.apply(latents, self, self.training)

    def _update(self, z: Tensor, idx: Tensor) -> None:
        """The EMA update from the batch `z` [B, D, H, W] and its indices, on the current stream, no host synchronisation."""
        E, cs, ea, prev = self.embedding.weight, self.cluster_size, self.embed_avg, self._pre_update
        for name, t in (("cluster_size", cs), ("embed_avg", ea), ("_pre_update", prev)):
            if t.device != z.device or t.dtype != torch.float32 or not t.is_contiguous():
                raise RuntimeError(f"movae_b200: VectorQuantizerEMA.{name} must be a contiguous float32 tensor on {z.device}")
        B, D, H, W = z.shape
        K = self.K
        stream = L.stream_of(z)
        lib = L.lib()
        ws = _buffer("ema", z.device, stream, lib.movae_vq_ema_workspace_bytes(B * H * W, K, D))
        with torch.cuda.device(z.device):
            if self.stats_reducer is None:
                L.check(lib.movae_vq_ema_update_f32(L.ptr(z), B, D, H * W, L.ptr(idx), K, self.decay, self.epsilon, L.ptr(E),
                                                    L.ptr(cs), L.ptr(ea), L.ptr(prev), L.ptr(ws), ws.numel(), stream),
                        "vq_ema_update_f32")
            else:
                if self._stats is None or self._stats.device != z.device:
                    self._stats = torch.empty(K + K * D, dtype=torch.float32, device=z.device)
                stats = self._stats
                L.check(lib.movae_vq_ema_stats_f32(L.ptr(z), B, D, H * W, L.ptr(idx), K, L.ptr(stats), L.ptr(ws), ws.numel(),
                                                   stream), "vq_ema_stats_f32")
                self.stats_reducer(stats)
                L.check(lib.movae_vq_ema_apply_f32(L.ptr(stats), K, D, self.decay, self.epsilon, L.ptr(E), L.ptr(cs), L.ptr(ea),
                                                   L.ptr(prev), L.ptr(ws), ws.numel(), L.stream_of(z)), "vq_ema_apply_f32")
        for t in (E, cs, ea, prev):                   # written through raw pointers: tell autograd
            torch.autograd.graph.increment_version(t)

    def extra_repr(self) -> str:
        return f"{self.K}, {self.D}, decay={self.decay}, epsilon={self.epsilon}"
