"""P-sharded aggregation across GPUs (one process per GPU, torch.distributed).

The Gramian is additive over column blocks of J (G = sum_s J_s J_s^T), the solve is k x k and the
recombination is column-local, so the whole multi-GPU path needs exactly ONE collective per step: an
all_reduce(sum) of the k x k float64 Gramian between K1 and K2 (SURVEY.md 8e).  Every rank then runs
K2 on bit-identical input and obtains identical weights.  The reference has no multi-device code;
this module is the host-side logic, and it is backend-agnostic so that it is testable with gloo.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib as L
from .aggregation import Aggregator


def shard_columns(P: int, rank: int, world: int, align: int = 4) -> Tuple[int, int]:
    """[lo, hi) column block of rank `rank`: contiguous, boundaries multiples of `align` columns
    (4 float32 = 16 bytes, so every shard keeps the float4 kernels), remainder on the last rank."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world size {world}")
    if P < 0 or align < 1:
        raise ValueError("P must be >= 0 and align >= 1")
    per = (P // world) // align * align
    lo = rank * per
    hi = P if rank == world - 1 else lo + per
    return lo, hi


def all_shards(P: int, world: int, align: int = 4) -> List[Tuple[int, int]]:
    return [shard_columns(P, r, world, align) for r in range(world)]


def gramian_allreduce(group: Optional[dist.ProcessGroup] = None) -> Callable[[torch.Tensor], None]:
    """In-place sum of the float64 [k, k] Gramian over the process group (<= 512 bytes: latency-bound)."""
    def reduce_(G: torch.Tensor) -> None:
        if G.dtype != torch.float64:
            raise TypeError("the Gramian exchanged between ranks must be float64")
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(G, op=dist.ReduceOp.SUM, group=group)
    return reduce_


def install_gramian_allreduce(aggregator: Aggregator, group: Optional[dist.ProcessGroup] = None) -> Aggregator:
    """Makes `aggregator(J_local)` aggregate the GLOBAL Jacobian whose column block this rank holds."""
    aggregator.weighting.gramian_reducer = gramian_allreduce(group)
    return aggregator


def codebook_allreduce(group: Optional[dist.ProcessGroup] = None) -> Callable[[torch.Tensor], None]:
    """In-place sum of a VectorQuantizerEMA's float32 [K + K*D] batch statistics (counts, then per-code sums) over the
    process group: one collective, capturable into a CUDA graph on NCCL."""
    def reduce_(stats: torch.Tensor) -> None:
        if stats.dtype != torch.float32:
            raise TypeError("the codebook statistics exchanged between ranks must be float32")
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return reduce_


def install_codebook_allreduce(vq, group: Optional[dist.ProcessGroup] = None):
    """Makes the EMA update of `vq` (a VectorQuantizerEMA) use the statistics of the GLOBAL batch when every rank
    quantizes its own slice of it: the counts and per-code sums are all-reduced between the statistics pass and the
    update (as the all_reduce in rosinality's `Quantize`), so the replicas apply the same update and their codebooks stay
    identical.  Returns `vq`."""
    if not hasattr(vq, "stats_reducer"):
        raise TypeError(f"install_codebook_allreduce needs a VectorQuantizerEMA, got {type(vq).__name__}")
    vq.stats_reducer = codebook_allreduce(group)
    return vq


def check_replicated(t: torch.Tensor, group: Optional[dist.ProcessGroup] = None) -> bool:
    """True when `t` (e.g. the weights, or MGDA's losses) is bit-identical on every rank."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return True
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
    return bool(torch.equal(lo, hi))


class P2PGramianExchange:
    """k x k Gramian exchange over NVLink peer memory, done INSIDE the fused aggregation kernel
    (include/movae_b200.h "P-sharded aggregation"): no collective launch on the per-step path, and -- the sequence
    number lives in the exchange buffer and is advanced by the kernel -- capturable into a CUDA graph.
    Construction is collective (all ranks of `group`, one GPU each, same node): every rank allocates an
    exchange buffer through the C ABI, the 64-byte CUDA IPC handles are all-gathered, peers are mapped."""

    def __init__(self, device: torch.device, group: Optional[dist.ProcessGroup] = None):
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("P2PGramianExchange needs an initialised torch.distributed process group")
        self.device = torch.device(device)
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if self.world > L.MAX_WORLD:
            raise RuntimeError(f"movae_b200: world size {self.world} > {L.MAX_WORLD} is not supported by this CUDA build")
        lib = L.lib()
        import ctypes
        self._own = ctypes.c_void_p()
        handle = ctypes.create_string_buffer(64)
        with torch.cuda.device(self.device):
            L.check(lib.movae_p2p_alloc(lib.movae_p2p_exchange_bytes(), ctypes.byref(self._own), handle), "p2p_alloc")
        mine = torch.tensor(list(handle.raw), dtype=torch.uint8, device=self.device)
        gathered = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(gathered, mine, group=group)
        self.ctx = L.P2PCtx(rank=self.rank, world=self.world)
        self._opened = []
        for r, t in enumerate(gathered):
            if r == self.rank:
                self.ctx.peers[r] = self._own.value
                continue
            peer = ctypes.c_void_p()
            with torch.cuda.device(self.device):
                L.check(lib.movae_p2p_open(bytes(t.cpu().tolist()), ctypes.byref(peer)), "p2p_open")
            self.ctx.peers[r] = peer.value
            self._opened.append(peer)
        self._status = torch.zeros(1, dtype=torch.int32, device=self.device)
        dist.barrier(group=group)

    def barrier(self) -> None:
        """Device-side barrier on the current stream (one tiny kernel over the peer flags, no host involvement, CUDA-graph
        capturable): after it the ranks' streams are aligned to within a flag round trip.  `barrier_failed()` reports a
        peer that never arrived."""
        import ctypes
        with torch.cuda.device(self.device):
            L.check(L.lib().movae_p2p_barrier(ctypes.byref(self.ctx), self._status.data_ptr(),
                                              torch.cuda.current_stream(self.device).cuda_stream), "p2p_barrier")

    def barrier_failed(self) -> bool:
        return bool(self._status.item())

    def close(self) -> None:
        lib = L.lib()
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            for p in self._opened:
                lib.movae_p2p_close(p)
            self._opened = []
            if self._own:
                lib.movae_p2p_free(self._own)
                self._own = None


class DataParallel:
    """Data-parallel Jacobian descent over one process per GPU (SURVEY.md 8e, "real DP training"): every rank holds a
    replica of the model and its own slice of the batch, so its Jacobian rows are gradients of LOCAL batch means.

    Instead of all-reducing k x P values and aggregating the full Jacobian redundantly on every rank, the rows are
    REDUCE-SCATTERED into contiguous 16-byte aligned column shards (one collective per row, averaged), each rank runs
    the fused aggregation launch on its shard -- the k x k float64 Gramian partials are exchanged inside it over peer
    memory (every rank then solves on bit-identical input) -- and the aggregated gradient is ALL-GATHERED: (k + 1) P values on the wire per rank
    instead of 2 k P, and K1 / K3 stream P / world columns.  Task-specific gradients (mtl_backward) are averaged by a
    plain all_reduce of their flat runs.  Attach with `DataParallel(aggregator)`; `backward` / `mtl_backward` pick
    it up from the aggregator.  The result equals single-process training on the concatenated batch when the shards
    have equal size.  Losses fed to `MGDA.set_losses` must already be the same on all ranks (all-reduce them)."""

    def __init__(self, aggregator: Aggregator, group: Optional[dist.ProcessGroup] = None, exchange: str = "auto"):
        """`exchange`: how the k x k Gramian partials of the column shards are summed -- "p2p" inside the fused
        aggregation kernel over NVLink peer memory (one launch per step, no collective; NCCL process groups on one
        node), "allreduce" through torch.distributed between K1 and K2 (any backend), "auto" = p2p when available."""
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("movae_b200.parallel.DataParallel needs an initialised torch.distributed process group")
        if exchange not in ("auto", "p2p", "allreduce"):
            raise ValueError(f"exchange must be 'auto', 'p2p' or 'allreduce', got {exchange!r}")
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.aggregator = aggregator
        self._native_rs = dist.get_backend(group) == "nccl"     # gloo (CPU tests of the plumbing) has no reduce_scatter
        use_p2p = exchange == "p2p" or (exchange == "auto" and self._native_rs and torch.cuda.is_available() and self.world > 1
                                        and self.world <= L.MAX_WORLD)
        self.exchange = None
        if use_p2p:
            self.exchange = install_p2p_gramian_exchange(aggregator, torch.device("cuda", torch.cuda.current_device()), group)
        else:
            install_gramian_allreduce(aggregator, group)
        if hasattr(aggregator.weighting, "draw_group"):          # PNUPGrad: every rank must use rank 0's per-step draw
            aggregator.weighting.draw_group = group if group is not None else True
        aggregator.data_parallel = self
        self._bufs: dict = {}

    def shard_len(self, P: int) -> int:
        """Columns per rank: P / world rounded up to 4 (every shard starts on a 16-byte boundary)."""
        per = (P + self.world - 1) // self.world
        return (per + 3) // 4 * 4

    def padded_columns(self, P: int) -> int:
        return self.shard_len(P) * self.world

    def _buf(self, name: str, shape, dtype, device) -> torch.Tensor:
        key = (name, tuple(shape), dtype, device)
        t = self._bufs.get(key)
        if t is None:
            t = torch.zeros(shape, dtype=dtype, device=device)
            self._bufs[key] = t
        return t

    # ---- row-wise reduce-scatter, overlapped with the backward passes that produce the following rows ------------------
    def begin_rows(self, k: int, P: int, dtype, device) -> None:
        """Start of a step: rows will be handed over one by one (autojac calls row_ready / row_zero as it fills J)."""
        self._Jsh = self._buf("Jsh", (k, self.shard_len(P)), dtype, device)
        self._works = []

    def row_ready(self, i: int, row_padded: torch.Tensor) -> None:
        """Row i of the padded Jacobian (world x shard columns) is complete on the current stream: its averaged
        reduce-scatter starts NOW, asynchronously, while autograd computes the next row."""
        Ps = self._Jsh.shape[1]
        if self._native_rs:
            self._works.append(dist.reduce_scatter_tensor(self._Jsh[i], row_padded, op=dist.ReduceOp.AVG, group=self.group,
                                                          async_op=True))
        else:
            tmp = row_padded.clone()
            dist.all_reduce(tmp, group=self.group)
            self._Jsh[i].copy_(tmp[self.rank * Ps:(self.rank + 1) * Ps] / self.world)

    def row_zero(self, i: int) -> None:
        """Row i is identically zero on every rank (an objective that never reaches the features): nothing on the wire."""
        self._Jsh[i].zero_()

    def finish_rows(self) -> torch.Tensor:
        for w in self._works:
            w.wait()                                             # the current stream waits for the collectives
        self._works = []
        return self._Jsh

    def reduce_scatter_rows(self, J_padded: torch.Tensor) -> torch.Tensor:
        """J_padded [k, world * Ps] (row stride arbitrary, columns beyond P zero) -> this rank's averaged shard [k, Ps]."""
        k, cols = J_padded.shape
        self._Jsh = self._buf("Jsh", (k, cols // self.world), J_padded.dtype, J_padded.device)
        self._works = []
        for i in range(k):
            self.row_ready(i, J_padded[i])
        return self.finish_rows()

    def all_gather_flat(self, g_shard: torch.Tensor) -> torch.Tensor:
        full = self._buf("gfull", (g_shard.numel() * self.world,), g_shard.dtype, g_shard.device)
        dist.all_gather_into_tensor(full, g_shard, group=self.group)
        return full

    def aggregate_rows_into(self, P: int, out: torch.Tensor, accumulate: bool) -> torch.Tensor:
        """After every row went through row_ready / row_zero: K1 on the shard, k x k all_reduce, K2 replicated, K3 on the
        shard, all-gather; `out` [P] is assigned or added to.  Returns the weights."""
        Jsh = self.finish_rows()
        g_shard = self._buf("gshard", (Jsh.shape[1],), Jsh.dtype, Jsh.device)
        # through the aggregator (not its bare weighting): COMFORT blends two solves, PNUPGrad draws, hooks fire
        w = self.aggregator.aggregate_into(Jsh, g_shard, accumulate=False)
        full = self.all_gather_flat(g_shard)
        if accumulate:
            out += full[:P]
        else:
            out.copy_(full[:P])
        return w

    def aggregate_into(self, J_padded: torch.Tensor, P: int, out: torch.Tensor, accumulate: bool) -> torch.Tensor:
        """The whole data-parallel aggregation of one step from a complete padded Jacobian."""
        self.reduce_scatter_rows(J_padded)
        return self.aggregate_rows_into(P, out, accumulate)

    def average_(self, tensors: List[torch.Tensor]) -> None:
        """In-place average over the ranks (task-specific gradients; flat runs when the parameters are flat)."""
        for t in tensors:
            if self._native_rs:
                dist.all_reduce(t, op=dist.ReduceOp.AVG, group=self.group)
            else:
                dist.all_reduce(t, group=self.group)
                t /= self.world


def install_p2p_gramian_exchange(aggregator: Aggregator, device: torch.device, group: Optional[dist.ProcessGroup] = None,
                                 exchange: Optional[P2PGramianExchange] = None) -> P2PGramianExchange:
    """Like install_gramian_allreduce, but the exchange happens inside the fused aggregation kernel (CUDA only).
    Replaces a previously installed torch.distributed reducer."""
    ex = exchange if exchange is not None else P2PGramianExchange(device, group)
    aggregator.weighting.gramian_reducer = None
    aggregator.weighting.p2p_exchange = ex
    if hasattr(aggregator.weighting, "draw_group"):
        aggregator.weighting.draw_group = group if group is not None else True
    return ex
