"""Flat parameter / gradient storage and the fused optimizer step (K7) -- SURVEY.md 8f rank 4.

The reference builds `optim.SGD | Adam | AdamW | RMSprop` over `net.parameters()`
(/root/reference/main.py:1169-1176), optionally clips with `clip_grad_norm_` (main.py:211-212) and calls
`optimizer.step()` (main.py:214).  Here the same four optimizers (same constructor keywords, same
`param_groups[0]["lr"]` contract for the LR schedulers of main.py:1179-1188, same `zero_grad()`) run as
ONE CUDA kernel over flat buffers:

  * `FlatParameters` re-homes every parameter into one flat float32 buffer (each tensor's offset
    rounded up to 4 elements = 16 bytes) and owns a flat gradient buffer of the same layout;
    `movae_b200.backward / mtl_backward` recognise such parameters and let K3 write the aggregated
    gradient straight into the flat gradient buffer (`.grad` = views of it), so aggregation ->
    clipping -> optimizer step never touches a per-tensor loop;
  * gradient clipping needs no pass over the gradients beyond one K1 launch (k = 1 Gramian = squared
    norm) and no host synchronisation;
  * the step count and the learning rate live on the device: the whole train step is CUDA-graph
    capturable (see `movae_b200.GraphedStep`).

CUDA-only, float32 parameters only; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes
import itertools
from typing import Iterable, List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib as L
from . import ops

_ALIGN = 4      # elements: every tensor starts on a 16-byte boundary of the flat buffers
_UIDS = itertools.count(1)


class FlatParameters:
    """One flat float32 buffer for the parameters and one for their gradients.

    After construction `p.data` of every parameter is a view of `flat_param`; `p.grad` is managed
    lazily: `None` after `zero_grad()` (torch's set_to_none default), a view of `flat_grad` once a
    gradient has been written for it."""

    def __init__(self, params: Iterable[Tensor]):
        seen, plist = set(), []
        for p in params:
            if id(p) in seen or not p.requires_grad:
                continue
            seen.add(id(p))
            plist.append(p)
        if not plist:
            raise ValueError("FlatParameters: no parameter requires grad")
        dev = plist[0].device
        for p in plist:
            L.require_cuda(p, "parameter")
            if p.dtype != torch.float32:
                raise TypeError(f"movae_b200: FlatParameters holds float32 parameters only (got {p.dtype})")
            if p.device != dev:
                raise RuntimeError("FlatParameters: all parameters must live on one CUDA device")
            if getattr(p, "_movae_flat", None) is not None:
                raise RuntimeError("FlatParameters: a parameter already belongs to another FlatParameters")
        self.params: List[Tensor] = plist
        self.uid = next(_UIDS)                     # identifies this layout in caches (id() can be recycled after garbage collection)
        self.offsets: List[int] = []
        off = 0
        for p in plist:
            self.offsets.append(off)
            off += (p.numel() + _ALIGN - 1) // _ALIGN * _ALIGN
        self.total = off
        self.device = dev
        self.flat_param = torch.zeros(self.total, dtype=torch.float32, device=dev)
        self.flat_grad = torch.zeros(self.total, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for i, p in enumerate(plist):
                view = self.flat_param[self.offsets[i]:self.offsets[i] + p.numel()].view(p.shape)
                view.copy_(p.data)
                p.data = view
                p._movae_flat = (self, i)
        self._grad_views: List[Tensor] = [self.flat_grad[o:o + p.numel()].view(p.shape) for o, p in zip(self.offsets, plist)]

    # ---- layout queries ----------------------------------------------------------------------------
    def padded_numel(self, i: int) -> int:
        return (self.params[i].numel() + _ALIGN - 1) // _ALIGN * _ALIGN

    def grad_view(self, p: Tensor) -> Tensor:
        return self._grad_views[p._movae_flat[1]]

    def grad_state(self, p: Tensor) -> str:
        """'none' | 'view' (p.grad IS the flat view) | 'other' (a gradient tensor living elsewhere)."""
        g = p.grad
        if g is None:
            return "none"
        v = self.grad_view(p)
        return "view" if (g.data_ptr() == v.data_ptr() and g.shape == v.shape and g.is_contiguous()) else "other"

    def plan(self, params: Sequence[Tensor]) -> Optional[Tuple[List[Tensor], List[int], int, int]]:
        """If `params` are exactly a run of consecutive tensors of this layout: (params in layout order,
        their column offsets relative to the run start, lo, hi) with [lo, hi) the run's range in the flat
        buffers (padding included); else None."""
        idx = sorted(p._movae_flat[1] for p in params)
        if not idx or len(set(idx)) != len(idx) or idx[-1] - idx[0] + 1 != len(idx):
            return None
        lo = self.offsets[idx[0]]
        hi = self.offsets[idx[-1]] + self.padded_numel(idx[-1])
        ordered = [self.params[i] for i in idx]
        return ordered, [self.offsets[i] - lo for i in idx], lo, hi

    def runs(self, indices: Iterable[int]) -> List[Tuple[int, int]]:
        """The [lo, hi) runs of the flat buffers (padding included) covered by the layout entries `indices`, each run
        merging consecutive entries."""
        runs: List[Tuple[int, int]] = []
        for i in sorted(indices):
            lo, hi = self.offsets[i], self.offsets[i] + self.padded_numel(i)
            if runs and runs[-1][1] == lo:
                runs[-1] = (runs[-1][0], hi)
            else:
                runs.append((lo, hi))
        return runs

    # ---- gradient management -----------------------------------------------------------------------
    def zero_grad(self, set_to_none: bool = True) -> None:
        if set_to_none:
            for p in self.params:
                p.grad = None
        else:
            self.flat_grad.zero_()
            for p, v in zip(self.params, self._grad_views):
                p.grad = v

    def adopt(self, params: Sequence[Tensor], grads: Sequence[Tensor]) -> None:
        """`p.grad = g` for parameters whose .grad is None, with g copied into the flat gradient buffer
        (one multi-tensor copy) so that `.grad` is a view of it."""
        dst, src = [], []
        for p, g in zip(params, grads):
            v = self.grad_view(p)
            dst.append(v)
            src.append(g.reshape(v.shape))
            p.grad = v
        if dst:
            torch._foreach_copy_(dst, src)

    def gather_grads(self) -> List[Tuple[int, int]]:
        """Makes every existing `.grad` a view of the flat gradient buffer (copying the ones that live
        elsewhere, e.g. after a plain `loss.backward()`), and returns the [lo, hi) runs of the flat
        buffers covered by parameters that HAVE a gradient (torch optimizers skip the others)."""
        dst, src, have = [], [], []
        for i, p in enumerate(self.params):
            st = self.grad_state(p)
            if st == "none":
                continue
            have.append(i)
            if st == "other":
                v = self._grad_views[i]
                dst.append(v)
                src.append(p.grad.detach().to(torch.float32).reshape(v.shape))
                p.grad = v
        if dst:
            torch._foreach_copy_(dst, src)
        return self.runs(have)


def flat_plan(params: Sequence[Tensor]):
    """(owner, ordered params, column offsets, lo, hi) when all `params` belong to one FlatParameters and
    form a consecutive run of its layout, else None (used by autojac)."""
    owner = None
    for p in params:
        info = getattr(p, "_movae_flat", None)
        if info is None:
            return None
        if owner is None:
            owner = info[0]
        elif owner is not info[0]:
            return None
    if owner is None:
        return None
    pl = owner.plan(params)
    if pl is None:
        return None
    ordered, cols, lo, hi = pl
    return owner, ordered, cols, lo, hi


class FusedOptimizer(torch.optim.Optimizer):
    """torch.optim.Optimizer whose `step()` is ONE launch of K7 over the flat buffers (per run of
    parameters that have a gradient: normally exactly one)."""

    _KIND = L.OPT_ADAM

    def __init__(self, params, defaults: dict, max_grad_norm: Optional[float] = None):
        self.flat = params if isinstance(params, FlatParameters) else FlatParameters(params)
        super().__init__(self.flat.params, defaults)
        if len(self.param_groups) != 1:
            raise ValueError("movae_b200 fused optimizers take one parameter group")
        self.max_grad_norm = max_grad_norm
        dev = self.flat.device
        n_state = L.lib().movae_optim_state_bytes()
        self._state = torch.zeros((n_state + 7) // 8, dtype=torch.int64, device=dev)      # step count lives here
        self._lr_dev = torch.full((1,), float(self.param_groups[0]["lr"]), dtype=torch.float64, device=dev)
        self._lr_host = float(self.param_groups[0]["lr"])
        self._gnorm_sq = torch.zeros((1, 1), dtype=torch.float64, device=dev)
        self._m: Optional[Tensor] = None
        self._v: Optional[Tensor] = None
        self.kernel_launches = 0

    # moment buffers are created by the subclasses (flat, same layout as the parameters)
    def _moments(self, first: bool, second: bool) -> None:
        z = lambda: torch.zeros(self.flat.total, dtype=torch.float32, device=self.flat.device)  # noqa: E731
        self._m = z() if first else None
        self._v = z() if second else None
        names = self._state_names()
        for o, p in zip(self.flat.offsets, self.flat.params):
            st = self.state[p]
            st["step"] = self._state[0]
            if self._m is not None:
                st[names[0]] = self._m[o:o + p.numel()].view(p.shape)
            if self._v is not None:
                st[names[1]] = self._v[o:o + p.numel()].view(p.shape)

    def _state_names(self) -> Tuple[str, str]:
        return "exp_avg", "exp_avg_sq"

    def _spec(self) -> L.OptimSpec:
        raise NotImplementedError

    @property
    def step_count(self) -> int:
        """Completed steps (reads the device counter: one D2H sync)."""
        return int(self._state[0].item())

    def sync_lr(self) -> None:
        """Pushes `param_groups[0]['lr']` to the device scalar the kernel reads (call after an LR scheduler
        step when `step()` itself is replayed from a CUDA graph)."""
        lr = float(self.param_groups[0]["lr"])
        if lr != self._lr_host:
            self._lr_dev.fill_(lr)
            self._lr_host = lr

    def state_dict(self):
        """torch.optim's format; `step` is exported the way torch's default (non-capturable) optimizers keep it -- a float32
        CPU scalar -- so the checkpoint loads into the matching torch optimizer too (one D2H read per checkpoint)."""
        sd = super().state_dict()
        step = torch.tensor(float(self.step_count), dtype=torch.float32)
        for st in sd["state"].values():
            if "step" in st:
                st["step"] = step.clone()
        return sd

    def load_state_dict(self, state_dict) -> None:
        """Accepts this class's own `state_dict()` (checkpointed at main.py:1407) and, the keys being torch.optim's
        ('step', 'exp_avg', 'exp_avg_sq' / 'momentum_buffer' / 'square_avg'), the matching torch optimizer's as well: the
        loaded tensors are copied INTO the flat moment buffers and the per-parameter state is re-linked to views of them."""
        super().load_state_dict(state_dict)
        names = self._state_names()
        step = None
        with torch.no_grad():
            for o, p in zip(self.flat.offsets, self.flat.params):
                st = self.state[p]
                for name, flat in ((names[0], self._m), (names[1], self._v)):
                    if flat is None:
                        continue
                    view = flat[o:o + p.numel()].view(p.shape)
                    if name in st and st[name] is not None and st[name].data_ptr() != view.data_ptr():
                        view.copy_(st[name])
                    st[name] = view
                if "step" in st:
                    step = int(st["step"]) if step is None else max(step, int(st["step"]))
                st["step"] = self._state[0]
            if step is not None:
                self._state[0] = step
        self._lr_host = float("nan")
        self.sync_lr()

    @torch.no_grad()
    def global_grad_norm_sq(self, runs: Optional[List[Tuple[int, int]]] = None) -> Tensor:
        """float64 [1,1] device tensor: squared L2 norm of all gradients (K1 with k = 1)."""
        runs = self.flat.gather_grads() if runs is None else runs
        first = True
        for lo, hi in runs:
            ops.gram(self.flat.flat_grad[lo:hi].view(1, -1), out=self._gnorm_sq, accumulate=not first)
            first = False
        if first:
            self._gnorm_sq.zero_()
        return self._gnorm_sq

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if not torch.cuda.is_current_stream_capturing():
            self.sync_lr()
        runs = self.flat.gather_grads()
        if not runs:
            return loss
        spec = self._spec()
        gn = 0
        if self.max_grad_norm is not None and self.max_grad_norm > 0:
            gn = self.global_grad_norm_sq(runs).data_ptr()
            spec.max_grad_norm = float(self.max_grad_norm)
        lib = L.lib()
        f = self.flat
        self.kernel_launches = 0
        with torch.cuda.device(f.device):
            stream = torch.cuda.current_stream(f.device).cuda_stream
            for r, (lo, hi) in enumerate(runs):
                off = 4 * lo
                spec.hold_step = int(r < len(runs) - 1)      # one optimizer step, however many launches
                L.check(lib.movae_optim_step_f32(f.flat_param.data_ptr() + off, f.flat_grad.data_ptr() + off,
                                                 (self._m.data_ptr() + off) if self._m is not None else 0,
                                                 (self._v.data_ptr() + off) if self._v is not None else 0,
                                                 hi - lo, ctypes.byref(spec), self._lr_dev.data_ptr(), gn,
                                                 self._state.data_ptr(), stream), "optim_step_f32")
                self.kernel_launches += 1
        # the kernel wrote the parameters through raw pointers: tell autograd (a backward pass over a graph retained from
        # BEFORE this step must raise torch's "modified by an inplace operation" error, not compute silently wrong
        # gradients).  The parameters keep their own version counters (`p.data = view` does not share the buffer's).
        torch._C._increment_version(f.params)
        return loss


class Adam(FusedOptimizer):
    """torch.optim.Adam(params, lr, betas, eps, weight_decay) as constructed at main.py:1172."""
    _KIND = L.OPT_ADAM

    def __init__(self, params, lr: float = 1e-3, betas: Tuple[float, float] = (0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.0, max_grad_norm: Optional[float] = None):
        if lr < 0 or eps < 0 or weight_decay < 0 or not (0 <= betas[0] < 1) or not (0 <= betas[1] < 1):
            raise ValueError("Invalid Adam hyper-parameter")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay), max_grad_norm)
        self._moments(True, True)

    def _spec(self) -> L.OptimSpec:
        g = self.param_groups[0]
        return L.OptimSpec(kind=self._KIND, lr=float(g["lr"]), beta1=g["betas"][0], beta2=g["betas"][1], eps=g["eps"],
                           weight_decay=g["weight_decay"], max_grad_norm=0.0)


class AdamW(Adam):
    """torch.optim.AdamW (decoupled weight decay, default 1e-2) as constructed at main.py:1174."""
    _KIND = L.OPT_ADAMW

    def __init__(self, params, lr: float = 1e-3, betas: Tuple[float, float] = (0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 1e-2, max_grad_norm: Optional[float] = None):
        super().__init__(params, lr, betas, eps, weight_decay, max_grad_norm)


class SGD(FusedOptimizer):
    """torch.optim.SGD(params, lr, momentum, weight_decay) as constructed at main.py:1170."""
    _KIND = L.OPT_SGD

    def __init__(self, params, lr: float = 1e-3, momentum: float = 0.0, weight_decay: float = 0.0,
                 max_grad_norm: Optional[float] = None):
        if lr < 0 or momentum < 0 or weight_decay < 0:
            raise ValueError("Invalid SGD hyper-parameter")
        super().__init__(params, dict(lr=lr, momentum=momentum, weight_decay=weight_decay), max_grad_norm)
        self._moments(momentum != 0, False)

    def _state_names(self):
        return "momentum_buffer", "unused"

    def _spec(self) -> L.OptimSpec:
        g = self.param_groups[0]
        return L.OptimSpec(kind=self._KIND, lr=float(g["lr"]), beta1=g["momentum"], beta2=0.0, eps=0.0,
                           weight_decay=g["weight_decay"], max_grad_norm=0.0)


class RMSprop(FusedOptimizer):
    """torch.optim.RMSprop(params, lr, alpha, eps, weight_decay) as constructed at main.py:1176."""
    _KIND = L.OPT_RMSPROP

    def __init__(self, params, lr: float = 1e-2, alpha: float = 0.99, eps: float = 1e-8, weight_decay: float = 0.0,
                 max_grad_norm: Optional[float] = None):
        if lr < 0 or eps < 0 or weight_decay < 0 or alpha < 0:
            raise ValueError("Invalid RMSprop hyper-parameter")
        super().__init__(params, dict(lr=lr, alpha=alpha, eps=eps, weight_decay=weight_decay), max_grad_norm)
        self._moments(False, True)

    def _state_names(self):
        return "unused", "square_avg"

    def _spec(self) -> L.OptimSpec:
        g = self.param_groups[0]
        return L.OptimSpec(kind=self._KIND, lr=float(g["lr"]), beta1=0.0, beta2=g["alpha"], eps=g["eps"],
                           weight_decay=g["weight_decay"], max_grad_norm=0.0)


def make_optimizer(name: str, params, lr: float, momentum: float = 0.9, weight_decay: float = 0.0,
                   max_grad_norm: Optional[float] = None) -> FusedOptimizer:
    """The optimizer factory of main.py:1169-1178 (`--optimizer sgd|adam|adamw|rmsprop`, `--lr`, `--momentum`, `--wd`)."""
    if name == "sgd":
        return SGD(params, lr=lr, momentum=momentum, weight_decay=weight_decay, max_grad_norm=max_grad_norm)
    if name == "adam":
        return Adam(params, lr=lr, weight_decay=weight_decay, max_grad_norm=max_grad_norm)
    if name == "adamw":
        return AdamW(params, lr=lr, weight_decay=weight_decay, max_grad_norm=max_grad_norm)
    if name == "rmsprop":
        return RMSprop(params, lr=lr, weight_decay=weight_decay, max_grad_norm=max_grad_norm)
    raise ValueError(f"Optimizer {name} not supported")


_PRE_REPLAY_SINK: Optional[list] = None


def register_pre_replay(callback) -> None:
    """Called (by code running under a GraphedStep capture) to register host work that must run before EVERY replay --
    per-step host state a captured launch can only read from device memory (PNUPGrad's random draw)."""
    if _PRE_REPLAY_SINK is None:
        raise RuntimeError("movae_b200: per-step host state can only be captured through movae_b200.GraphedStep "
                           "(a bare torch.cuda.graph capture would freeze it)")
    _PRE_REPLAY_SINK.append(callback)


class GraphedStep:
    """Captures one whole train step (zero_grad -> forward -> backward / mtl_backward -> optimizer step) into a
    CUDA graph and replays it: the BASELINE model configs are launch-bound (hundreds of ~5 us kernels per step),
    and nothing on the movae_b200 path synchronises with the host, so the step is capturable as is.

    `fn` must be capture-safe: static input tensors (refill them in place before each replay), no `.item()` /
    `.cpu()` inside, optimizers whose step count lives on the device (the fused ones here, or torch's with
    `capturable=True`).  `fn` runs `warmup` times eagerly on a side stream first (lazy initialisation, cuDNN
    algorithm selection, workspace allocation), then once under capture; its return value (tensors living in
    the graph's memory pool) is returned by every replay.

    With `parallel.DataParallel` the NCCL collectives of the step are captured too (validated on 2 GPUs: identical
    replicas after replay); set TORCH_NCCL_ASYNC_ERROR_HANDLING=0 before `init_process_group`, and do not call
    `destroy_process_group()` while the graph is alive (it blocks): drop the graph first or just exit."""

    def __init__(self, fn, warmup: int = 3):
        if not torch.cuda.is_available():
            raise RuntimeError("movae_b200.GraphedStep needs a CUDA device (there is no CPU fallback)")
        self.fn = fn
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        global _PRE_REPLAY_SINK
        self.graph = torch.cuda.CUDAGraph()
        self._pre_replay: list = []
        _PRE_REPLAY_SINK = self._pre_replay
        try:
            with torch.cuda.graph(self.graph):
                self.outputs = fn()
        finally:
            _PRE_REPLAY_SINK = None
        # The captured launches hold raw addresses of the package's cached buffers (Jacobian, Gramian / quantizer
        # workspaces, K6 scratch).  Those caches may later REPLACE an entry (a bigger batch, another model): keep the
        # tensors that exist now alive for as long as this graph does, so a replay never touches freed memory.
        from . import autojac, ops as _ops, quantizer as _q

        self._keepalive = (list(autojac._J_CACHE.values()) + list(autojac._ZEROS.values()) + list(_ops._workspaces.values()) +
                           list(_q._buffers.values()))
        self.replays = 0

    def __call__(self):
        for cb in self._pre_replay:
            cb()
        self.graph.replay()
        self.replays += 1
        return self.outputs
