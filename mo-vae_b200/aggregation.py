"""Host-side mirror of the reference's aggregator API over the CUDA kernels.

Same names, constructor kwargs, call shape and error behaviour as the reference so that
`/root/reference/main.py:1191-1250` works unchanged with these classes:

    agg(J[k,P]) -> g[P]                      (torchjd Aggregator.forward; call sites main.py:189-196)
    agg.weighting : nn.Module, J[k,P] -> w[k]  (forward hooks `(module, (J,), w)`, main.py:1248-1250)
    UPGrad(pref_vector=None, norm_eps=1e-4, reg_eps=1e-4, solver="quadprog")       (main.py:1195)
    AlignedMTL(pref_vector=None, scale_mode="min"|"median"|"rmse")     (aligned_mtl.py:56-63)
    MGDA(norm_type, epsilon, max_iters, stable, min_eigenvalue_eps), .set_losses(), .mgda_weighting
                                                                      (mgda.py:89-131)
    Sum(), Mean()                                                     (main.py:1198, :1223-1224)
    PCGrad(), IMTLG()                                                 (torchjd; selectable at main.py:1196-1220)

Every call is ONE fused launch (Gramian pass over J, small solve by the last CTA to arrive, recombination
pass + write-back; csrc/aggregate.cu) on the current CUDA stream with no host synchronisation -- or, when a
torch.distributed `gramian_reducer` is installed, K1 -> reducer -> K2 -> K3; diagnostics that the reference gets
through `.item()` (MGDA convergence_count / gamma, the gradient-similarity hook) stay on the device
in `weighting.last_diag` and are only fetched when somebody reads them.
"""
from __future__ import annotations

from typing import Callable, Literal, Optional

import torch
from torch import Tensor, nn

from . import _lib as L
from . import ops

_NormType = Literal["none", "l2", "loss", "loss+"]


class Weighting(nn.Module):
    """Maps a Jacobian J[k,P] to weights w[k] through its Gramian.

    On its own (`weighting(J)`, what a hook-less caller or torchjd's WeightedAggregator does) it runs the fused kernel
    without its recombination phase: Gramian pass + solve in ONE launch.  When its aggregator has just run the whole
    fused step for the same J, the weights of that launch are handed over instead of being recomputed, so the forward
    hooks the reference registers here (main.py:1248-1250) still fire with `(module, (J,), w)`."""

    def __init__(self):
        super().__init__()
        self.last_gramian: Optional[Tensor] = None   # float64 [k,k] on the device (summed over the ranks when P-sharded)
        self.last_diag: Optional[Tensor] = None      # float64 [8] on the device (include/movae_b200.h)
        # in-place reduction applied to the float64 Gramian between K1 and K2 (any torch.distributed backend; what the
        # gloo CPU tests of the plumbing use).  Setting it selects the three-launch path K1 -> reducer -> K2 -> K3.
        self.gramian_reducer: Optional[Callable[[Tensor], None]] = None
        # fused alternative: the k x k exchange happens INSIDE the fused kernel over NVLink peer memory
        # (parallel.P2PGramianExchange); no collective launch at all
        self.p2p_exchange = None
        self._handover = None                         # (w, diag, G) of the aggregator's fused launch for the next forward

    def solve_spec(self, k: int):
        """(movae_solve_spec, pref-or-losses tensor | None, device aux tensor | None) for the C entry points."""
        raise NotImplementedError

    def prepare_step(self, device, k: Optional[int] = None) -> None:
        """Host-side per-step state that must reach the device BEFORE the launch of a k-row aggregation (PNUPGrad's and
        PCGrad's draws).  Default: nothing."""

    def _select(self, w: Tensor, k: int) -> Tensor:
        """The weights this module reports out of the solve's output vector."""
        return w[:k]

    def from_gramian(self, gramian: Tensor) -> Tensor:
        """Weights from an already reduced float64 Gramian (K2 only)."""
        spec, vec, aux = self.solve_spec(gramian.shape[0])
        w, diag = ops.solve(gramian, spec, vec, aux)
        self.last_gramian, self.last_diag = gramian, diag
        return self._select(w, gramian.shape[0])

    def forward(self, matrix: Tensor) -> Tensor:
        if self._handover is not None:
            w, self.last_diag, self.last_gramian = self._handover
            self._handover = None
            return w
        ops.check_jacobian(matrix)
        matrix = matrix.detach()
        self.prepare_step(matrix.device, matrix.shape[0])
        if self.gramian_reducer is not None:
            G = ops.gram(matrix)
            self.gramian_reducer(G)
            return self.from_gramian(G)
        k = matrix.shape[0]
        spec, vec, aux = self.solve_spec(k)
        w, diag, G, _ = ops.aggregate(matrix, spec, vec, aux, exchange=self.p2p_exchange, want_grad=False)
        self.last_gramian, self.last_diag = G, diag
        return self._select(w, k)

    # -- lazily fetched diagnostics (each read is one D2H sync, on demand only) -----------------
    def _diag(self, slot: int) -> float:
        if self.last_diag is None:
            raise RuntimeError("no aggregation has run yet")
        return float(self.last_diag[slot].item())

    @property
    def gradient_similarity(self) -> float:
        """cos(J^T w, mean_rows(J)) -- what the hook main.py:94-122 recomputes with two passes over J."""
        return self._diag(L.DIAG_SIMILARITY)

    def check_status(self) -> None:
        """Synchronising check of the device-side status word of the last solve.  torchjd raises ValueError when quadprog
        returns None; a peer of the P-sharded exchange that never delivered its Gramian partial raises RuntimeError (its
        text contains "CUDA", so the skip-batch handler of main.py:197-208 matches).  The weights of such a step are NaN."""
        st = self._diag(L.DIAG_STATUS)
        if st == 2.0:
            raise RuntimeError("movae_b200: CUDA peer-memory Gramian exchange timed out (a rank did not publish its partial)")
        if st != 0.0:
            raise ValueError(f"Failed to solve the quadratic programming problem (KKT residual "
                             f"{self._diag(L.DIAG_RESIDUAL):.3e}, or non-finite weights).")


class Aggregator(nn.Module):
    """g = weighting(J) @ J as ONE fused launch (Gramian pass, solve, recombination + write-back)."""

    def __init__(self, weighting: Weighting):
        super().__init__()
        self.weighting = weighting

    def forward(self, matrix: Tensor) -> Tensor:
        out = torch.empty(matrix.shape[1] if matrix.dim() == 2 else 0, dtype=torch.float32, device=matrix.device)
        self.aggregate_into(matrix, out)
        return out

    def _fused(self, matrix: Tensor, out: Tensor, accumulate: bool):
        """One launch; returns (weights used for the recombination, weights the weighting reports to its hooks)."""
        wt = self.weighting
        k = matrix.shape[0]
        wt.prepare_step(matrix.device, k)
        spec, vec, aux = wt.solve_spec(k)
        w, diag, G, _ = ops.aggregate(matrix, spec, vec, aux, out=out, accumulate=accumulate, exchange=wt.p2p_exchange)
        return w[:k], (wt._select(w, k), diag, G)

    def supports_segments(self) -> bool:
        """True when the aggregation can run over a segmented Jacobian (`aggregate_segments_into`): the fused launch is in
        use and nobody needs to SEE a [k, P] matrix -- forward hooks on the weighting receive `(module, (J,), w)`
        (main.py:1248-1250), so a hooked weighting keeps the flat-J path."""
        wt = self.weighting
        return wt.gramian_reducer is None and not wt._forward_hooks and not wt._forward_pre_hooks

    def aggregate_segments_into(self, rows, numels, out_offsets, out: Tensor, accumulate: bool = False) -> Tensor:
        """The fused launch over the gradient tensors themselves (ops.aggregate_segments): no flat Jacobian is built."""
        wt = self.weighting
        k = len(rows)
        dev = rows[0][0].device
        wt.prepare_step(dev, k)
        spec, vec, aux = wt.solve_spec(k)
        w, diag, G = ops.aggregate_segments(rows, numels, out_offsets, spec, vec, aux, out, accumulate, exchange=wt.p2p_exchange)
        wt.last_gramian, wt.last_diag = G, diag
        return w[:k]

    def aggregate_into(self, matrix: Tensor, out: Tensor, accumulate: bool = False) -> Tensor:
        """K3 writes (or adds) straight into `out`, the flat buffer the parameters' .grad tensors are views of.
        Returns the weights."""
        ops.check_jacobian(matrix)
        matrix = matrix.detach()            # the aggregation is non-differentiable (nupgrad.py:83)
        wt = self.weighting
        if wt.gramian_reducer is not None:  # three launches around a torch.distributed reduction of the Gramian
            w = wt(matrix)
            ops.recombine(matrix, w, out=out, accumulate=accumulate)
            return w
        w, wt._handover = self._fused(matrix, out, accumulate)
        wt(matrix)                          # hands the launch's weights to the forward hooks, no kernel
        return w


GramianWeightedAggregator = Aggregator


# ---- Sum / Mean ----------------------------------------------------------------------------------
class _ConstantWeighting(Weighting):
    def __init__(self, value: Optional[float]):
        super().__init__()
        self._value = value      # None -> 1/k

    def solve_spec(self, k: int):
        return L.SolveSpec(kind=L.SOLVE_CONSTANT, value=-1.0 if self._value is None else self._value), None, None


class Sum(Aggregator):
    """torchjd `Sum` (selectable as `jd_sum`, main.py:1223-1224): w = 1."""

    def __init__(self):
        super().__init__(_ConstantWeighting(1.0))

    def __repr__(self) -> str:
        return "Sum()"


class Mean(Aggregator):
    """torchjd `Mean` (main.py:1198): w = 1/k."""

    def __init__(self):
        super().__init__(_ConstantWeighting(None))

    def __repr__(self) -> str:
        return "Mean()"


# ---- UPGrad ---------------------------------------------------------------------------------------
class UPGradWeighting(Weighting):
    norm_mode = "trace"          # torchjd `normalize`: divide the Gramian by its trace

    def __init__(self, pref_vector: Optional[Tensor], norm_eps: float, reg_eps: float, solver: str):
        super().__init__()
        if solver != "quadprog":
            raise ValueError(f"Unknown solver {solver!r}; only 'quadprog' semantics are implemented")
        self._pref_vector = pref_vector
        self.norm_eps = norm_eps
        self.reg_eps = reg_eps
        self.solver = solver

    def _norm_mode(self) -> str:
        return self.norm_mode

    def solve_spec(self, k: int):
        return (L.SolveSpec(kind=L.SOLVE_UPGRAD, mode=L.UPGRAD_NORM[self._norm_mode()], norm_eps=self.norm_eps,
                            reg_eps=self.reg_eps), self._pref_vector, None)


class UPGrad(Aggregator):
    """Drop-in for torchjd.aggregation.UPGrad as constructed at main.py:1195."""

    def __init__(self, pref_vector: Optional[Tensor] = None, norm_eps: float = 0.0001, reg_eps: float = 0.0001,
                 solver: Literal["quadprog"] = "quadprog"):
        super().__init__(UPGradWeighting(pref_vector, norm_eps, reg_eps, solver))
        self._pref_vector = pref_vector
        self._norm_eps = norm_eps
        self._reg_eps = reg_eps
        self._solver = solver

    def __repr__(self) -> str:
        return (f"{self.__class__.__name__}(pref_vector={self._pref_vector!r}, norm_eps={self._norm_eps}, "
                f"reg_eps={self._reg_eps}, solver={self._solver!r})")


class DualProjWeighting(UPGradWeighting):
    """torchjd `_DualProjWrapper`: w = project_weights(u, regularize(normalize(G))) with u the preference weights (1/k)."""

    def solve_spec(self, k: int):
        return L.SolveSpec(kind=L.SOLVE_DUALPROJ, norm_eps=self.norm_eps, reg_eps=self.reg_eps), self._pref_vector, None


class DualProj(Aggregator):
    """Drop-in for torchjd.aggregation.DualProj as constructed at main.py:1221-1222."""

    def __init__(self, pref_vector: Optional[Tensor] = None, norm_eps: float = 0.0001, reg_eps: float = 0.0001,
                 solver: Literal["quadprog"] = "quadprog"):
        super().__init__(DualProjWeighting(pref_vector, norm_eps, reg_eps, solver))
        self._pref_vector = pref_vector
        self._norm_eps = norm_eps
        self._reg_eps = reg_eps
        self._solver = solver

    def __repr__(self) -> str:
        return (f"{self.__class__.__name__}(pref_vector={self._pref_vector!r}, norm_eps={self._norm_eps}, "
                f"reg_eps={self._reg_eps}, solver={self._solver!r})")


class _NUPGradWeighting(UPGradWeighting):
    """utils/torchmoo/nupgrad.py:122-126: UPGrad on the Gramian rescaled to the smallest gradient norm."""
    norm_mode = "min_l2"


class NUPGrad(Aggregator):
    """Drop-in for utils/torchmoo/nupgrad.py:37 `NUPGrad` (main.py:1226)."""

    def __init__(self, pref_vector: Optional[Tensor] = None, norm_eps: float = 0.0001, reg_eps: float = 0.0001,
                 solver: Literal["quadprog"] = "quadprog"):
        super().__init__(_NUPGradWeighting(pref_vector, norm_eps, reg_eps, solver))
        self._pref_vector, self._norm_eps, self._reg_eps, self._solver = pref_vector, norm_eps, reg_eps, solver

    def __repr__(self) -> str:
        return (f"{self.__class__.__name__}(pref_vector={self._pref_vector!r}, norm_eps={self._norm_eps}, "
                f"reg_eps={self._reg_eps}, solver={self._solver!r})")


class _HostDraw:
    """Mixin of the weightings whose solve consumes a per-aggregation draw from torch's default HOST generator, consumed
    exactly as the reference consumes it.  The outcome is written into a fixed device buffer (`_aux`) that the solve reads
    as d_aux, with stream-ordered writes, so a CUDA-graph replay follows the draws too: under capture the draw is deferred
    to `GraphedStep`'s pre-replay callbacks (the captured launch only reads the buffer, which one eager run must have
    created).  P-sharded / data-parallel: rank 0's draw is broadcast (`draw_group`, set by parallel.py; any installed
    Gramian exchange implies the default group), all ranks must solve the same problem."""
    _aux: Optional[Tensor] = None
    draw_group = None                           # a process group (or True = the default one) whose rank 0's draw every rank uses

    def _draw_into_device(self, device, k: Optional[int]) -> None:
        raise NotImplementedError

    def _device_buffer(self, n: int, device) -> Tensor:
        if self._aux is None or self._aux.device != torch.device(device) or self._aux.numel() != n:
            self._aux = torch.zeros(n, dtype=torch.float32, device=device)
        return self._aux

    def _broadcast_draw(self) -> None:
        grp = self.draw_group
        if grp is None and (self.p2p_exchange is not None or self.gramian_reducer is not None):
            grp = True
        if grp is not None:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size(None if grp is True else grp) > 1:
                dist.broadcast(self._aux, src=0, group=None if grp is True else grp)

    def prepare_step(self, device, k: Optional[int] = None) -> None:
        if torch.cuda.is_current_stream_capturing():
            if self._aux is None:
                raise RuntimeError(f"movae_b200: run {self._draw_owner} once eagerly before capturing it into a CUDA graph")
            from .optim import register_pre_replay
            register_pre_replay(lambda: self._draw_into_device(device, k))   # every replayed step draws on the host first
            return
        self._draw_into_device(device, k)


class _PNUPGradWeighting(_HostDraw, UPGradWeighting):
    """utils/torchmoo/pnupgrad.py:127-134: with probability `prob` the cosine-normalised Gramian G / (|g_i||g_j|),
    otherwise NUPGrad's; the draw is `torch.rand(1).item() < prob` on the HOST RNG exactly like the reference, once per
    aggregation.  Its outcome is a device flag the solve reads (MOVAE_UPGRAD_NORM_DRAW; _HostDraw carries it under CUDA
    graphs and across ranks)."""
    _draw_owner = "PNUPGrad"

    def __init__(self, pref_vector, prob: float, norm_eps: float, reg_eps: float, solver: str):
        super().__init__(pref_vector, norm_eps, reg_eps, solver)
        self.prob = prob
        self._mode = "min_l2"

    def _norm_mode(self) -> str:
        return "draw"

    def draw(self, device=None) -> str:
        """One host draw; updates the device flag (a fill kernel carrying the value as an argument: race-free)."""
        self._mode = "l2" if torch.rand(1).item() < self.prob else "min_l2"
        if device is not None:
            self._device_buffer(1, device).fill_(1.0 if self._mode == "l2" else 0.0)
            self._broadcast_draw()
        return self._mode

    def _draw_into_device(self, device, k: Optional[int]) -> None:
        self.draw(device)

    def solve_spec(self, k: int):
        spec, vec, _ = super().solve_spec(k)
        return spec, vec, self._aux


class PNUPGrad(Aggregator):
    """Drop-in for utils/torchmoo/pnupgrad.py:37 `PNUPGrad` (main.py:1228)."""

    def __init__(self, pref_vector: Optional[Tensor] = None, prob: float = 0.5, norm_eps: float = 0.0001,
                 reg_eps: float = 0.0001, solver: Literal["quadprog"] = "quadprog"):
        super().__init__(_PNUPGradWeighting(pref_vector, prob, norm_eps, reg_eps, solver))
        self._pref_vector, self._prob, self._norm_eps, self._reg_eps, self._solver = pref_vector, prob, norm_eps, reg_eps, solver

    def __repr__(self) -> str:
        return (f"{self.__class__.__name__}(pref_vector={self._pref_vector!r}, prob={self._prob}, norm_eps={self._norm_eps}, "
                f"reg_eps={self._reg_eps}, solver={self._solver!r})")


# ---- PCGrad / IMTL-G ------------------------------------------------------------------------------------
class PCGradWeighting(_HostDraw, Weighting):
    """torchjd `PCGradWeighting` [torchjd-recall] as a weighting of the Gramian: chain i starts at e_i and, in the order of
    a fresh `torch.randperm(k)`, removes its conflict with every other row j (c_j -= <g_j, J^T c> / |g_j|^2 when that is
    negative); w = the sum of the k chains, all float32 like torchjd's CPU loop.  The k permutations are drawn on the HOST
    RNG exactly as torchjd draws them (k `torch.randperm(k)` calls per aggregation, row i first for chain i) and reach the
    solve as a k x k device table."""
    _draw_owner = "PCGrad"

    def __init__(self):
        super().__init__()
        self.last_perms: Optional[Tensor] = None     # int64 [k, k] CPU: the permutations of the last draw

    def draw(self, k: int, device=None) -> Tensor:
        """One aggregation's draw: k `torch.randperm(k)` calls; with `device`, the table is copied into the device buffer
        the solve reads (stream-ordered, from pinned memory the caching host allocator keeps until the copy has run)."""
        self.last_perms = torch.stack([torch.randperm(k) for _ in range(k)])
        if device is not None:
            src = self.last_perms.to(torch.float32).reshape(-1).pin_memory()
            self._device_buffer(k * k, device).copy_(src, non_blocking=True)
            self._broadcast_draw()
        return self.last_perms

    def _draw_into_device(self, device, k: Optional[int]) -> None:
        if k is None:
            raise ValueError("movae_b200: PCGrad draws k permutations per aggregation; prepare_step needs k")
        self.draw(k, device)

    def solve_spec(self, k: int):
        if self._aux is None or self._aux.numel() != k * k:
            raise RuntimeError(f"movae_b200: no PCGrad permutation table for k={k} on the device (call prepare_step first)")
        return L.SolveSpec(kind=L.SOLVE_PCGRAD), None, self._aux


class PCGrad(Aggregator):
    """Drop-in for torchjd.aggregation.PCGrad (selectable as `pcgrad`, main.py:1196-1220)."""

    def __init__(self):
        super().__init__(PCGradWeighting())

    def __repr__(self) -> str:
        return "PCGrad()"


class IMTLGWeighting(Weighting):
    """torchjd `IMTLGWeighting` [torchjd-recall]: v = pinv(G) sqrt(diag G), w = v / sum(v) (zeros when |sum(v)| < 1e-12),
    the pseudo-inverse from a float64 eigen-decomposition with pinv's default tolerance (k eps32 max|eigenvalue|)."""

    def solve_spec(self, k: int):
        return L.SolveSpec(kind=L.SOLVE_IMTLG), None, None

    @property
    def rank(self) -> int:
        """Eigenvalues of the Gramian the pseudo-inverse kept in the last solve."""
        return int(self._diag(L.DIAG_RANK))


class IMTLG(Aggregator):
    """Drop-in for torchjd.aggregation.IMTLG (selectable as `imtlg`, main.py:1196-1220)."""

    def __init__(self):
        super().__init__(IMTLGWeighting())

    def __repr__(self) -> str:
        return "IMTLG()"


# ---- Aligned-MTL ------------------------------------------------------------------------------------
class AlignedMTLWeighting(Weighting):
    def __init__(self, pref_vector: Optional[Tensor] = None, scale_mode: str = "min"):
        super().__init__()
        self._pref_vector = pref_vector
        self._scale_mode = scale_mode

    def solve_spec(self, k: int):
        if self._scale_mode not in L.AMTL_SCALE:     # raised at call time like aligned_mtl.py:127-130
            raise ValueError(f"Invalid scale_mode={self._scale_mode!r}. Expected 'min', 'median', or 'rmse'.")
        return L.SolveSpec(kind=L.SOLVE_ALIGNED_MTL, mode=L.AMTL_SCALE[self._scale_mode]), self._pref_vector, None

    @property
    def rank(self) -> int:
        return int(self._diag(L.DIAG_RANK))


class AlignedMTL(Aggregator):
    """Drop-in for utils/torchmoo/aligned_mtl.py:39 `AlignedMTL`."""

    def __init__(self, pref_vector: Optional[Tensor] = None, scale_mode: Literal["min", "median", "rmse"] = "min"):
        super().__init__(AlignedMTLWeighting(pref_vector, scale_mode=scale_mode))
        self._pref_vector = pref_vector
        self._scale_mode = scale_mode

    def __repr__(self) -> str:
        return f"{self.__class__.__name__}(pref_vector={self._pref_vector!r}, scale_mode={self._scale_mode!r})"


# ---- MGDA ------------------------------------------------------------------------------------------------
def _check_norm_type(norm_type: str) -> None:
    if norm_type not in ("none", "l2", "loss", "loss+"):
        raise ValueError(f"Parameter `norm_type` should be 'none', 'l2', 'loss', or 'loss+'. Found "
                         f"`norm_type = {norm_type!r}`.")


class MGDAWeighting(Weighting):
    """Drop-in for utils/torchmoo/mgda.py:156 `MGDAWeighting` (Frank-Wolfe runs inside K2)."""

    def __init__(self, norm_type: _NormType = "none", epsilon: float = 1e-5, max_iters: int = 250,
                 stable: bool = False, min_eigenvalue_eps: float = 1e-10):
        super().__init__()
        _check_norm_type(norm_type)
        self.norm_type = norm_type
        self.epsilon = epsilon
        self.max_iters = max_iters
        self.stable = stable
        self.min_eigenvalue_eps = min_eigenvalue_eps
        self._losses: Optional[Tensor] = None
        # set by COMFORT: device float32 {1 - beta, beta}; the solve then also runs UPGrad and blends (MOVAE_SOLVE_COMFORT)
        self._comfort_coef: Optional[Tensor] = None
        self._comfort_eps = (0.0, 0.0)

    def set_losses(self, losses: Tensor) -> None:
        if losses.dim() != 1:
            raise ValueError(f"Parameter `losses` should be a 1D tensor. Found `losses.shape = {losses.shape}`.")
        self._losses = losses.detach()

    def _checked_losses(self, n: int) -> Optional[Tensor]:
        if self.norm_type not in ("loss", "loss+"):
            return None
        if self._losses is None:
            raise RuntimeError(f"Losses must be set before calling forward() when using "
                               f"norm_type={self.norm_type!r}. Call set_losses() first.")
        if self._losses.shape[0] != n:
            raise ValueError(f"Number of losses ({self._losses.shape[0]}) must match the number of rows in "
                             f"the gramian ({n}).")
        return self._losses

    def solve_spec(self, k: int):
        comfort = self._comfort_coef is not None
        spec = L.SolveSpec(kind=L.SOLVE_COMFORT if comfort else L.SOLVE_MGDA, mode=L.MGDA_NORM[self.norm_type],
                           max_iters=self.max_iters, stable=int(self.stable), epsilon=self.epsilon,
                           min_eigenvalue_eps=self.min_eigenvalue_eps, norm_eps=self._comfort_eps[0], reg_eps=self._comfort_eps[1])
        return spec, self._checked_losses(k), self._comfort_coef

    def _select(self, w: Tensor, k: int) -> Tensor:
        # under COMFORT the solve returns [blend, w_mgda]; this module (where the reference's hooks sit, comfort.py:131) is MGDA
        return w[k:2 * k] if self._comfort_coef is not None else w[:k]

    @property
    def convergence_count(self) -> Optional[int]:
        return None if self.last_diag is None else int(self._diag(L.DIAG_COUNT))

    @property
    def gamma(self) -> Optional[float]:
        return None if self.last_diag is None else self._diag(L.DIAG_GAMMA)


class MGDA(Aggregator):
    """Drop-in for utils/torchmoo/mgda.py:12 `MGDA` (`isinstance(aggregator, MGDA)` is tested at
    main.py:185 before `set_losses`)."""

    def __init__(self, norm_type: _NormType = "none", epsilon: float = 1e-5, max_iters: int = 250,
                 stable: bool = False, min_eigenvalue_eps: float = 1e-10):
        _check_norm_type(norm_type)
        mgda_weighting = MGDAWeighting(norm_type=norm_type, epsilon=epsilon, max_iters=max_iters, stable=stable,
                                       min_eigenvalue_eps=min_eigenvalue_eps)
        super().__init__(mgda_weighting)
        self._mgda_weighting = mgda_weighting
        self._norm_type = norm_type
        self._epsilon = epsilon
        self._max_iters = max_iters
        self._stable = stable

    @property
    def mgda_weighting(self) -> MGDAWeighting:
        return self._mgda_weighting

    def set_losses(self, losses: Tensor) -> None:
        self._mgda_weighting.set_losses(losses)

    def __repr__(self) -> str:
        return (f"{self.__class__.__name__}(norm_type={self._norm_type!r}, epsilon={self._epsilon}, "
                f"max_iters={self._max_iters}, stable={self._stable})")


def StableMGDA(norm_type: _NormType = "none", epsilon: float = 1e-5, max_iters: int = 250,
               min_eigenvalue_eps: float = 1e-10) -> MGDA:
    """mgda.py:140-153."""
    return MGDA(norm_type=norm_type, epsilon=epsilon, max_iters=max_iters, stable=True,
                min_eigenvalue_eps=min_eigenvalue_eps)


# ---- COMFORT ------------------------------------------------------------------------------------------
def beta_schedule(epoch: int, total_epochs: int, k: float = 1.0, a: float = 1.0, l: float = 0.01, u: float = 1.0) -> float:  # noqa: E741
    """utils/torchmoo/comfort.py:26-65: beta rises from `l` (first epoch) to `u` (last epoch)."""
    import math

    if total_epochs <= 1:
        return u
    progress = (epoch - 1) / (total_epochs - 1)
    progress = min(1.0, max(0.0, progress)) ** a
    f = progress if k <= 0 else (1.0 - math.exp(-k * progress)) / (1.0 - math.exp(-k))
    return float(min(u, max(l, l + (u - l) * f)))


class COMFORT:
    """Drop-in for utils/torchmoo/comfort.py:68 `COMFORT`: (1 - beta) MGDA(J) + beta UPGrad(J).
    The recombination is linear in the weights, so ONE fused launch (one Gramian pass, both solves inside the solve phase,
    one recombination pass with w = (1 - beta) w_mgda + beta w_upgrad) replaces the reference's two full aggregations.
    beta lives in DEVICE memory (`set_epoch` rewrites it), so a step captured into a CUDA graph follows the schedule."""

    def __init__(self, mgda_norm_type: _NormType = "none", mgda_stable: bool = False, mgda_epsilon: float = 1e-5,
                 mgda_max_iters: int = 250, mgda_min_eigenvalue_eps: float = 1.0, beta_k: float = 1.0, beta_a: float = 1.0,
                 beta_l: float = 0.01, beta_u: float = 1.0):
        self._mgda = MGDA(norm_type=mgda_norm_type, epsilon=mgda_epsilon, max_iters=mgda_max_iters, stable=mgda_stable,
                          min_eigenvalue_eps=mgda_min_eigenvalue_eps)
        self._upgrad = UPGrad()
        self._beta_k, self._beta_a, self._beta_l, self._beta_u = beta_k, beta_a, beta_l, beta_u
        self._current_epoch = 1
        self._total_epochs = 1
        self._norm_type = mgda_norm_type
        self.weighting = self._mgda.mgda_weighting            # hooks attach here, like the reference (comfort.py:131)
        self.weighting._comfort_eps = (self._upgrad.weighting.norm_eps, self._upgrad.weighting.reg_eps)
        self._coef: Optional[Tensor] = None

    def set_epoch(self, epoch: int, total_epochs: int) -> None:
        self._current_epoch, self._total_epochs = epoch, total_epochs
        if self._coef is not None:
            self._write_coef()

    def set_losses(self, losses: Tensor) -> None:
        self._mgda.set_losses(losses)

    def _get_beta(self) -> float:
        return beta_schedule(self._current_epoch, self._total_epochs, k=self._beta_k, a=self._beta_a, l=self._beta_l,
                             u=self._beta_u)

    def _write_coef(self) -> None:
        beta = self._get_beta()
        # two fills carrying the float64-rounded-once coefficients as kernel arguments (not captured: set_epoch runs
        # between steps); the reference multiplies float32 tensors by the Python floats (1.0 - beta) and beta
        self._coef[0:1].fill_(1.0 - beta)
        self._coef[1:2].fill_(beta)

    def _ensure_coef(self, device) -> None:
        if self._coef is None or self._coef.device != torch.device(device):
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("movae_b200: run COMFORT once eagerly before capturing it into a CUDA graph")
            self._coef = torch.zeros(2, dtype=torch.float32, device=device)
            self._write_coef()
            self.weighting._comfort_coef = self._coef

    def blended_weights(self, matrix: Tensor) -> Tensor:
        """K1 + both solves (one launch, no recombination): the blended weights; fires the MGDA weighting's hooks."""
        ops.check_jacobian(matrix)
        matrix = matrix.detach()
        self._ensure_coef(matrix.device)
        wt = self.weighting
        k = matrix.shape[0]
        if wt.gramian_reducer is not None:
            G = ops.gram(matrix)
            wt.gramian_reducer(G)
            spec, vec, aux = wt.solve_spec(k)
            w, diag = ops.solve(G, spec, vec, aux)
        else:
            spec, vec, aux = wt.solve_spec(k)
            w, diag, G, _ = ops.aggregate(matrix, spec, vec, aux, exchange=wt.p2p_exchange, want_grad=False)
        wt._handover = (w[k:2 * k], diag, G)
        wt(matrix)
        return w[:k]

    def __call__(self, matrix: Tensor) -> Tensor:
        out = torch.empty(matrix.shape[1] if matrix.dim() == 2 else 0, dtype=torch.float32, device=matrix.device)
        self.aggregate_into(matrix, out)
        return out

    supports_segments = Aggregator.supports_segments

    def aggregate_segments_into(self, rows, numels, out_offsets, out: Tensor, accumulate: bool = False) -> Tensor:
        self._ensure_coef(rows[0][0].device)
        return Aggregator.aggregate_segments_into(self, rows, numels, out_offsets, out, accumulate)

    def aggregate_into(self, matrix: Tensor, out: Tensor, accumulate: bool = False) -> Tensor:
        ops.check_jacobian(matrix)
        matrix = matrix.detach()
        self._ensure_coef(matrix.device)
        wt = self.weighting
        k = matrix.shape[0]
        if wt.gramian_reducer is not None:
            w = self.blended_weights(matrix)
            ops.recombine(matrix, w, out=out, accumulate=accumulate)
            return w
        spec, vec, aux = wt.solve_spec(k)
        w, diag, G, _ = ops.aggregate(matrix, spec, vec, aux, out=out, accumulate=accumulate, exchange=wt.p2p_exchange)
        wt._handover = (w[k:2 * k], diag, G)
        wt(matrix)
        return w[:k]

    def __repr__(self) -> str:
        return (f"COMFORT(mgda={self._mgda!r}, beta_k={self._beta_k}, beta_a={self._beta_a}, beta_l={self._beta_l}, "
                f"beta_u={self._beta_u})")


# ---- name map of the training driver ----------------------------------------------------------------
def make_aggregator(name: Optional[str], *, agg_norm_eps: float = 1e-4, agg_reg_eps: float = 1e-4,
                    mgda_epsilon: float = 1e-5, mgda_max_iters: int = 250, pref_weights=None):
    """Aggregator factory with the reference's `--aggregator` names (main.py:1191-1246) for the
    aggregators on the hot path.  Returns None / "sum" exactly where the reference does."""
    if name is None:
        return None
    n = name.lower()
    if n == "sum":
        return "sum"            # plain total_loss.backward(), no Jacobian (main.py:176-177)
    if n == "upgrad":
        return UPGrad(norm_eps=agg_norm_eps, reg_eps=agg_reg_eps, pref_vector=pref_weights)
    if n == "mean":
        return Mean()
    if n == "jd_sum":
        return Sum()
    if n in ("aligned_mtl", "aligned_mtl_min", "amtl", "amtl_min"):
        return AlignedMTL(pref_vector=pref_weights)
    if n == "aligned_mtl_median":
        return AlignedMTL(scale_mode="median", pref_vector=pref_weights)
    if n == "aligned_mtl_rmse":
        return AlignedMTL(scale_mode="rmse", pref_vector=pref_weights)
    if n == "mgda":
        return MGDA(epsilon=mgda_epsilon, max_iters=mgda_max_iters)
    if n == "mgda_ln":
        return MGDA(epsilon=mgda_epsilon, max_iters=mgda_max_iters, norm_type="l2")
    if n == "mgda_gn":
        return MGDA(epsilon=mgda_epsilon, max_iters=mgda_max_iters, norm_type="loss")
    if n == "mgda_lgn":
        return MGDA(epsilon=mgda_epsilon, max_iters=mgda_max_iters, norm_type="loss+")
    if n == "dualproj":
        return DualProj(norm_eps=agg_norm_eps, reg_eps=agg_reg_eps)
    if n == "nupgrad":
        return NUPGrad(norm_eps=agg_norm_eps, reg_eps=agg_reg_eps)
    if n == "pnupgrad":
        return PNUPGrad(norm_eps=agg_norm_eps, reg_eps=agg_reg_eps)
    if n == "comfort":
        return COMFORT(mgda_epsilon=mgda_epsilon, mgda_max_iters=mgda_max_iters, mgda_min_eigenvalue_eps=1e-10)
    if n == "pcgrad":
        return PCGrad()
    if n == "imtlg":
        return IMTLG()
    if n in ("cagrad", "nashmtl"):
        # selectable in the reference (main.py:1196-1220) but outside this path: CAGrad solves a cone program over the
        # simplex (its result hangs on that solver's tolerances), NashMTL keeps optimiser state across steps
        raise ValueError(f"Aggregator {name} not supported by movae_b200 (not on the Gramian-weighting hot path); "
                         f"use torchjd.aggregation for it")
    raise ValueError(f"Aggregator {name} not supported")
