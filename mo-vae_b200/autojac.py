"""Jacobian-descent engine entry points with the signatures the reference calls
(/root/reference/main.py:17, :189-196):

    backward(tensors, aggregator=..., inputs=None, retain_graph=False)
    mtl_backward(losses=, features=, aggregator=, tasks_params=None, shared_params=None, retain_graph=False)

They replace torchjd.autojac.{backward,mtl_backward} (un-vendored dependency, requirements.txt:58;
semantics restated in SURVEY.md App. A).  The k per-objective backward passes are plain torch
autograd (not ours); what changes is everything after them:

  * NO Jacobian matrix is built at all (SURVEY 8f rank 1): the fused kernel reads every objective's gradient of every
    shared parameter tensor where autograd left it, through a table of k row pointers per tensor
    (`movae_aggregate_segments_f32`) -- no per-parameter reshape + `torch.cat`, not even one copy.  The flat
    J[k, ldJ] buffer (one multi-tensor copy per row) remains for the cases that need a matrix: a data-parallel plan
    (the rows are reduce-scattered), forward hooks on the weighting (they receive J), more than 32 shared tensors;
  * Gramian pass, solve and recombination are ONE launch on the current stream;
  * K3 writes the aggregated gradient into one flat buffer and the parameters' `.grad` become views
    of it (assign if `.grad is None`, `+=` otherwise: torchjd `Accumulate` semantics).  When the
    parameters live in a `movae_b200.FlatParameters` (optim.py) that buffer is the persistent flat
    gradient buffer the fused optimizer step (K7) reads, and J's columns follow its 16-byte aligned layout;
  * `mtl_backward` back-propagates only the objectives that reach the features at all: a loss whose
    feature gradients are all `None` (e.g. `embedding_loss`, vq_vae.py:52) is an identically zero row
    of J and costs one memset instead of a backward pass through the shared encoder.
"""
from __future__ import annotations

from typing import Callable, Iterable, Iterator, List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from .aggregation import Aggregator
from .optim import flat_plan

_J_CACHE: dict = {}


def _leaves_of(roots: Sequence[Tensor], stop_at: Sequence[Tensor] = ()) -> List[Tensor]:
    """Leaf tensors requiring grad in the autograd graph of `roots`, in discovery order (DFS over
    grad_fn.next_functions).  Traversal does not descend below the grad_fns of `stop_at`."""
    stop = {t.grad_fn for t in stop_at if t.grad_fn is not None}
    seen, out, out_ids = set(), [], set()
    stack = [t.grad_fn for t in reversed(list(roots)) if t.grad_fn is not None]
    for t in roots:
        if t.grad_fn is None and t.requires_grad and id(t) not in out_ids:
            out.append(t)
            out_ids.add(id(t))
    while stack:
        fn = stack.pop()
        if fn is None or fn in seen:
            continue
        seen.add(fn)
        if hasattr(fn, "variable"):                       # AccumulateGrad node -> leaf
            v = fn.variable
            if v.requires_grad and id(v) not in out_ids:
                out.append(v)
                out_ids.add(id(v))
            continue
        if fn in stop:
            continue
        for nxt, _ in reversed(fn.next_functions):
            if nxt is not None and nxt not in seen:
                stack.append(nxt)
    return out


def _jacobian_buffer(k: int, P: int, device: torch.device, layout: tuple = (), min_ld: int = 0) -> Tensor:
    """The flat J[k, ldJ] buffer, zero-filled at allocation (padding columns of an aligned layout are never
    written afterwards, so they stay zero) and reused every step for the same (k, layout).  `min_ld`: a data-parallel
    aggregation wants the row padded to world x shard columns (parallel.DataParallel)."""
    ld = max((P + 3) // 4 * 4, min_ld)
    key = (device, k, ld, layout)
    buf = _J_CACHE.get(key)
    if buf is None:
        _J_CACHE.clear()                                  # one live model per process is the norm
        buf = torch.zeros((k, ld), dtype=torch.float32, device=device)
        _J_CACHE[key] = buf
    return buf[:, :P] if ld != P else buf


def _dense_offsets(params: Sequence[Tensor]) -> List[int]:
    offs, off = [], 0
    for p in params:
        offs.append(off)
        off += p.numel()
    return offs


def _fill_row(J: Tensor, i: int, params: Sequence[Tensor], grads: Sequence[Optional[Tensor]], offsets: Sequence[int]) -> None:
    dst, src = [], []
    for p, g, off in zip(params, grads, offsets):
        view = J[i, off:off + p.numel()]
        if g is None:
            view.zero_()
        else:
            dst.append(view)
            src.append(g.reshape(-1))
    if dst:
        torch._foreach_copy_(dst, src)


def _row_gradients(outputs: Sequence, params: Sequence[Tensor], grad_outputs_per_row: Sequence[Optional[Sequence[Tensor]]],
                   retain_graph: bool) -> Iterator[Tuple[int, Optional[Sequence[Optional[Tensor]]]]]:
    """Yields (i, grads) in row order: the tuple autograd returns for d(sum_j <outputs[j], grad_outputs_per_row[i][j]>) / d params
    (entries may be None), or None for an identically zero row (no backward pass).  `outputs[i]` is row i's own list when
    every row differentiates its own scalar (`backward`).  Row i's pass runs when the consumer asks for it, so whatever
    the consumer does with row i-1 is enqueued before it."""
    # One backward pass per row.  One vmapped pass over all rows (torchjd's default) measured slower on every BASELINE model
    # config, per step under a CUDA graph on one B200 (power limit not recorded): 2.64 / 15.97 / 23.11 ms against
    # 2.57 / 14.98 / 21.92 ms for VQ-VAE / GG-VQ-VAE / VQ-VAE2 -- the vmapped convolution backward costs more than the
    # launches it saves.
    per_row = isinstance(outputs[0], (list, tuple))
    last = max((i for i, g in enumerate(grad_outputs_per_row) if g is not None), default=-1)
    for i, g in enumerate(grad_outputs_per_row):
        if g is None:
            yield i, None
        else:
            yield i, torch.autograd.grad(outputs[i] if per_row else outputs, params, grad_outputs=list(g),
                                         retain_graph=retain_graph or i < last, allow_unused=True)


def _fill_jacobian(J: Tensor, rows, params: Sequence[Tensor], offsets: Sequence[int], dp=None) -> None:
    """J[i] from row i's gradients (an identically zero row is one memset).  With a data-parallel plan (`dp`) every
    finished row is handed to it before the next row's backward pass runs, so its reduce-scatter overlaps that pass."""
    if dp is not None:
        k, P = J.shape
        padded = dp.padded_columns(P)
        Jp = J.as_strided((k, padded), (J.stride(0) if k > 1 else padded, 1))
        dp.begin_rows(k, P, J.dtype, J.device)
    for i, grads in rows:
        if grads is None:
            J[i].zero_()
        else:
            _fill_row(J, i, params, grads, offsets)
        if dp is not None:
            if grads is None:
                dp.row_zero(i)
            else:
                dp.row_ready(i, Jp[i])


_ZEROS: dict = {}


def _zero_row(device: torch.device, n: int) -> Tensor:
    """A shared all-zero buffer every identically zero Jacobian entry points at (never written)."""
    z = _ZEROS.get(device)
    if z is None or z.numel() < n:
        z = torch.zeros(max(n, 1 << 16), dtype=torch.float32, device=device)
        _ZEROS[device] = z
    return z


def _segment_rows(rows, params: Sequence[Tensor]) -> List[List[Tensor]]:
    """Every row as the list of gradient tensors the segmented launch reads in place; a missing gradient, and every entry
    of an identically zero row, is the shared zero buffer."""
    from . import ops

    zero = _zero_row(params[0].device, max(p.numel() for p in params))
    out = []
    for _, gs in rows:
        if gs is None:
            out.append([zero] * len(params))
            continue
        r = []
        for g in gs:
            if g is None:
                r.append(zero)
            else:
                g = g.detach()
                r.append(g if ops.segment_ok(g) else g.to(torch.float32).contiguous().clone())     # rare: a strided / unaligned gradient
        out.append(r)
    return out


def _segments_possible(params: Sequence[Tensor], aggregator) -> bool:
    from . import _lib as L

    return (_dp_of(aggregator) is None and len(params) <= L.MAX_SEGMENTS
            and hasattr(aggregator, "supports_segments") and aggregator.supports_segments())


def _write_back(params: Sequence[Tensor], cols: Sequence[int], P: int, plan, launch: Callable[[Tensor, bool], Tensor]) -> None:
    """torchjd's Accumulate rule for the aggregated gradient: `launch(out, accumulate)` writes (or adds) it into `out`, with
    params[j] at columns cols[j]..cols[j]+numel, and each `.grad` is assigned when None, added to otherwise.  When the
    parameters are a run of a FlatParameters layout (`plan`; `cols` are then its columns) and every `.grad` is None, or
    every `.grad` is already its view, `out` is the persistent flat gradient buffer the fused optimizer step (K7) reads;
    otherwise it is a fresh buffer of P columns."""
    if plan is not None:
        owner, _, _, lo, hi = plan
        states = {owner.grad_state(p) for p in params}
        if states == {"none"}:
            launch(owner.flat_grad[lo:hi], False)
            for p in params:
                p.grad = owner.grad_view(p)
            return
        if states == {"view"}:
            launch(owner.flat_grad[lo:hi], True)
            return
    flat = torch.empty(P, dtype=torch.float32, device=params[0].device)
    launch(flat, False)
    add_dst, add_src = [], []
    for p, off in zip(params, cols):
        g = flat[off:off + p.numel()].view(p.shape)
        if p.grad is None:
            p.grad = g
        else:
            add_dst.append(p.grad)
            add_src.append(g)
    if add_dst:
        torch._foreach_add_(add_dst, add_src)


def _check_aggregator(aggregator) -> None:
    if not isinstance(aggregator, Aggregator) and not hasattr(aggregator, "aggregate_into"):
        raise TypeError(f"aggregator must be a movae_b200 Aggregator, got {type(aggregator).__name__}")


def _dp_of(aggregator):
    return getattr(aggregator, "data_parallel", None)


def _run_aggregation(J: Tensor, aggregator: Aggregator, out: Tensor, accumulate: bool) -> Tensor:
    """K1 -> K2 -> K3 into `out`; through the reduce-scatter / all-gather plan when the aggregator is data-parallel."""
    dp = _dp_of(aggregator)
    if dp is None:
        return aggregator.aggregate_into(J, out, accumulate=accumulate)
    return dp.aggregate_rows_into(J.shape[1], out, accumulate)     # the rows were handed over while they were built


def _layout(params: Sequence[Tensor]):
    """(params in J's column order, column offsets, P, plan, cache key)."""
    plan = flat_plan(params)
    if plan is not None:
        _, ordered, cols, lo, hi = plan
        return ordered, cols, hi - lo, plan, ("flat", plan[0].uid, lo, hi)
    params = list(params)
    return params, _dense_offsets(params), sum(p.numel() for p in params), None, ()


def _aggregate_rows(outputs: Sequence, params: Sequence[Tensor], grad_outputs_per_row: Sequence[Optional[Sequence[Tensor]]],
                    retain_graph: bool, aggregator) -> None:
    """The rows of `_row_gradients` aggregated into the parameters' `.grad`: by the segmented launch over the gradient
    tensors themselves when nothing needs a [k, P] matrix, else through the flat J."""
    params, cols, P, plan, key = _layout(params)
    if P == 0:
        return
    rows = _row_gradients(outputs, params, grad_outputs_per_row, retain_graph)
    if _segments_possible(params, aggregator):
        numels = [p.numel() for p in params]
        seg = _segment_rows(rows, params)
        if plan is None:                                  # every tensor on a 16-byte boundary, as a FlatParameters layout has it
            cols, P = [], 0
            for n in numels:
                cols.append(P)
                P += (n + 3) // 4 * 4
        _write_back(params, cols, P, plan, lambda out, acc: aggregator.aggregate_segments_into(seg, numels, cols, out, accumulate=acc))
        return
    dp = _dp_of(aggregator)
    J = _jacobian_buffer(len(grad_outputs_per_row), P, params[0].device, key, dp.padded_columns(P) if dp else 0)
    _fill_jacobian(J, rows, params, cols, dp)
    _write_back(params, cols, P, plan, lambda out, acc: _run_aggregation(J, aggregator, out, acc))


def backward(tensors: Sequence[Tensor] | Tensor, aggregator: Aggregator, inputs: Optional[Iterable[Tensor]] = None,
             retain_graph: bool = False, parallel_chunk_size: Optional[int] = None) -> None:
    """Jacobian of `tensors` (k scalar losses) w.r.t. `inputs` (default: every leaf that requires
    grad in their graph), aggregated into `.grad` (main.py:196).  `parallel_chunk_size` is accepted for torchjd's
    signature and ignored: the rows are always k sequential backward passes."""
    _check_aggregator(aggregator)
    losses = [tensors] if isinstance(tensors, Tensor) else list(tensors)
    if len(losses) == 0:
        raise ValueError("`tensors` cannot be empty")
    for t in losses:
        if t.numel() != 1:
            raise ValueError("movae_b200.backward supports scalar objectives only (one Jacobian row each)")
    params = list(inputs) if inputs is not None else _leaves_of(losses)
    if not params:
        return
    # every row differentiates ITS OWN loss: a stacked loss with one-hot cotangents would walk the union graph of all
    # objectives k times and push zero cotangents through the other objectives' private subgraphs (0 * inf = NaN)
    outputs = [[t.reshape(())] for t in losses]
    ones = [[torch.ones((), dtype=t.dtype, device=t.device)] for t in losses]
    _aggregate_rows(outputs, params, ones, retain_graph, aggregator)


def mtl_backward(losses: Sequence[Tensor], features: Sequence[Tensor] | Tensor, aggregator: Aggregator,
                 tasks_params: Optional[Sequence[Iterable[Tensor]]] = None,
                 shared_params: Optional[Iterable[Tensor]] = None, retain_graph: bool = False,
                 parallel_chunk_size: Optional[int] = None) -> None:
    """Multi-task variant (main.py:188-194): task-specific parameters receive the plain SUM of
    their losses' gradients; the shared parameters (those the features depend on) receive the
    aggregation of the k rows  d loss_i / d shared  obtained by back-propagating each loss's
    feature gradients through the shared part.  `parallel_chunk_size` is accepted for torchjd's signature and ignored."""
    _check_aggregator(aggregator)
    losses = list(losses)
    feats = [features] if isinstance(features, Tensor) else list(features)
    if len(losses) == 0:
        raise ValueError("`losses` cannot be empty")
    if len(feats) == 0:
        raise ValueError("`features` cannot be empty")
    shared = list(shared_params) if shared_params is not None else _leaves_of(feats)
    shared_ids = {id(p) for p in shared}
    if tasks_params is None:
        tasks = [[p for p in _leaves_of([l], stop_at=feats) if id(p) not in shared_ids] for l in losses]
    else:
        tasks = [list(tp) for tp in tasks_params]
        if len(tasks) != len(losses):
            raise ValueError("`tasks_params` must have one entry per loss")

    dp = _dp_of(aggregator)
    feat_grads: List[Optional[List[Tensor]]] = []
    task_sum: dict = {}                                  # id(param) -> [param, this call's gradient summed over the tasks]
    for loss, tparams in zip(losses, tasks):
        outs = torch.autograd.grad(loss, feats + tparams, retain_graph=True, allow_unused=True)
        fg = outs[:len(feats)]
        if all(g is None for g in fg):
            feat_grads.append(None)                       # this objective never reaches the features: zero row of J
        else:
            feat_grads.append([torch.zeros_like(f) if g is None else g for f, g in zip(feats, fg)])
        for p, g in zip(tparams, outs[len(feats):]):
            if g is None:
                continue
            ent = task_sum.get(id(p))
            if ent is None:
                task_sum[id(p)] = [p, g]
            else:
                ent[1] = ent[1] + g
    # task-specific parameters: the plain SUM of their losses' gradients (averaged over the ranks when data-parallel),
    # assigned when .grad is None (into the flat gradient buffer if the parameter lives in one), else added
    fresh_flat: dict = {}
    for p, g in task_sum.values():
        if p.grad is None and getattr(p, "_movae_flat", None) is not None:
            ent = fresh_flat.setdefault(id(p._movae_flat[0]), [p._movae_flat[0], [], []])
            ent[1].append(p)
            ent[2].append(g)
        else:
            if dp is not None:
                g = g.contiguous() if g._base is None else g.clone()
                dp.average_([g])
            if p.grad is None:
                p.grad = g.clone() if g._base is not None else g
            else:
                p.grad += g
    for owner, ps, gs in fresh_flat.values():
        owner.adopt(ps, gs)
        if dp is not None:
            dp.average_([owner.flat_grad[lo:hi] for lo, hi in owner.runs(p._movae_flat[1] for p in ps)])
    _aggregate_rows(feats, shared, feat_grads, retain_graph, aggregator)
