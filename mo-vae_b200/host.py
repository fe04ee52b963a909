"""Aggregation of a Jacobian that lives in HOST memory (the `e2e` leg of bench.py): the C-ABI
host pipeline streams J to the GPU in column chunks overlapped with K1, solves on the device, and
streams K3's output back.  A P-sharded caller passes `gramian_reducer` (one k x k allreduce)."""
from __future__ import annotations

import ctypes
from typing import Callable, Optional

import torch

from . import _lib as L
from . import ops
from .aggregation import Aggregator


class HostAggregationPlan:
    """Owns the device staging buffers for one (k, P) so repeated steps do not allocate.

    `run` is synchronous (returns when `h_out` is complete).  `run_async` / `wait` pipeline consecutive steps over
    `depth` sets of device buffers: while step i's aggregated gradient is still on its way to the host (device-to-host
    copies on a stream of their own), step i + 1's Jacobian is already streaming in -- PCIe is full duplex, and the
    host-to-device direction (4kP bytes) is the longer one, so the per-step cost drops from H2D + D2H to H2D."""

    def __init__(self, k: int, P: int, device: torch.device, chunk_cols: int = 1 << 22, depth: int = 2):
        if not (1 <= k <= L.MAX_K):
            raise RuntimeError(f"movae_b200: k={k} objectives outside 1..{L.MAX_K} is not supported by this CUDA build")
        self.k, self.P, self.device = k, P, torch.device(device)
        self.ld = (P + 3) // 4 * 4
        self.chunk_cols = max(4, chunk_cols // 4 * 4)
        self.depth = max(1, depth)
        self._sets = None
        self._alloc(1)
        self.copy_stream = torch.cuda.Stream(device=device)
        self.d2h_stream = torch.cuda.Stream(device=device)
        self.kernel_launches = 0
        self._issued = 0
        self._done: list = []

    def _alloc(self, n: int) -> None:
        k, dev = self.k, self.device
        sets = self._sets or []
        while len(sets) < n:
            sets.append({"J": torch.empty((k, self.ld), dtype=torch.float32, device=dev),
                         "grad": torch.empty(self.ld, dtype=torch.float32, device=dev),
                         "G": torch.zeros((k, k), dtype=torch.float64, device=dev),
                         "w": torch.empty(2 * k, dtype=torch.float32, device=dev),      # COMFORT reports two weight vectors
                         "diag": torch.empty(L.DIAG_DOUBLES, dtype=torch.float64, device=dev)})
        self._sets = sets
        self.d_J, self.d_grad, self.d_G, self.d_w, self.d_diag = (sets[0][n_] for n_ in ("J", "grad", "G", "w", "diag"))

    def _check(self, h_J: torch.Tensor, h_out: torch.Tensor) -> None:
        k, P = self.k, self.P
        if h_J.is_cuda or h_out.is_cuda:
            raise ValueError("aggregate_host expects HOST tensors")
        if h_J.shape != (k, P) or h_J.dtype != torch.float32 or h_J.stride(1) != 1:
            raise ValueError(f"h_J must be float32 [{k},{P}] with contiguous rows")
        if h_out.shape != (P,) or h_out.dtype != torch.float32 or not h_out.is_contiguous():
            raise ValueError(f"h_out must be contiguous float32 [{P}]")

    def _enqueue(self, h_J, aggregator, h_out, gramian_reducer, bufs, synchronous: bool):
        k, P = self.k, self.P
        lib = L.lib()
        with torch.cuda.device(self.device):
            cs = torch.cuda.current_stream(self.device)
            ws = ops._gram_workspace(self.device, k, cs.cuda_stream)
            L.check(lib.movae_host_gram_f32(h_J.data_ptr(), k, P, h_J.stride(0) if k > 1 else max(P, 1),
                                            bufs["J"].data_ptr(), self.ld, bufs["G"].data_ptr(), ws.data_ptr(), ws.numel(),
                                            self.chunk_cols, cs.cuda_stream, self.copy_stream.cuda_stream), "host_gram_f32")
            if gramian_reducer is not None:
                gramian_reducer(bufs["G"])
            if hasattr(aggregator, "_ensure_coef"):
                aggregator._ensure_coef(self.device)          # COMFORT: the blend coefficients live on the device
            aggregator.weighting.prepare_step(self.device, k)
            spec, vec, aux = aggregator.weighting.solve_spec(k)
            vec = ops._dev_f32(vec, self.device, k, "pref_vector/losses")
            L.check(lib.movae_solve_aux(bufs["G"].data_ptr(), k, ctypes.byref(spec), L.ptr(vec), L.ptr(aux), bufs["w"].data_ptr(),
                                        bufs["diag"].data_ptr(), cs.cuda_stream), "solve")
            if synchronous:
                L.check(lib.movae_host_recombine_f32(bufs["J"].data_ptr(), k, P, self.ld, bufs["w"].data_ptr(),
                                                     bufs["grad"].data_ptr(), h_out.data_ptr(), self.chunk_cols,
                                                     cs.cuda_stream, self.copy_stream.cuda_stream), "host_recombine_f32")
            else:
                L.check(lib.movae_host_recombine_async_f32(bufs["J"].data_ptr(), k, P, self.ld, bufs["w"].data_ptr(),
                                                           bufs["grad"].data_ptr(), h_out.data_ptr(), self.chunk_cols,
                                                           cs.cuda_stream, self.d2h_stream.cuda_stream), "host_recombine_async_f32")
        aggregator.weighting.last_gramian, aggregator.weighting.last_diag = bufs["G"], bufs["diag"]
        n_chunks = (P + self.chunk_cols - 1) // self.chunk_cols
        self.kernel_launches = 2 * n_chunks + 1

    def run(self, h_J: torch.Tensor, aggregator: Aggregator, h_out: torch.Tensor,
            gramian_reducer: Optional[Callable[[torch.Tensor], None]] = None) -> torch.Tensor:
        self._check(h_J, h_out)
        self.wait()
        self._enqueue(h_J, aggregator, h_out, gramian_reducer, self._sets[0], synchronous=True)
        return h_out

    def run_async(self, h_J: torch.Tensor, aggregator: Aggregator, h_out: torch.Tensor,
                  gramian_reducer: Optional[Callable[[torch.Tensor], None]] = None) -> None:
        """Enqueues one step and returns; `h_out` is complete after `wait()`.  At most `depth` steps are in flight: the
        call blocks on the step that last used this step's device buffers.  `h_J` must stay untouched until the step's
        host-to-device copies have run (i.e. until the next-but-`depth` call returns, or `wait()`)."""
        self._check(h_J, h_out)
        self._alloc(self.depth)
        slot = self._issued % self.depth
        while len(self._done) >= self.depth:
            self._done.pop(0).synchronize()
        self._enqueue(h_J, aggregator, h_out, gramian_reducer, self._sets[slot], synchronous=False)
        ev = torch.cuda.Event()
        ev.record(self.d2h_stream)
        self._done.append(ev)
        self._issued += 1

    def wait(self) -> None:
        """Blocks until every step issued with `run_async` has delivered its result to the host."""
        while self._done:
            self._done.pop(0).synchronize()


def aggregate_host(h_J: torch.Tensor, aggregator: Aggregator, h_out: Optional[torch.Tensor] = None,
                   device: str | torch.device = "cuda", plan: Optional[HostAggregationPlan] = None) -> torch.Tensor:
    """One-shot convenience wrapper: host J[k,P] -> host g[P] (synchronous)."""
    k, P = h_J.shape
    plan = plan or HostAggregationPlan(k, P, torch.device(device))
    if h_out is None:
        h_out = torch.empty(P, dtype=torch.float32, pin_memory=True)
    return plan.run(h_J, aggregator, h_out)
