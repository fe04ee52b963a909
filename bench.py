#!/usr/bin/env python
"""bench.py -- headline benchmark of the MO-VAE hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl movae|reference] [--k 3] [--P 100000000] [--agg upgrad]
                    [--scaling weak|strong] [--quick] [--dump-outputs DIR] [--detail-dir DIR]

Workload (BASELINE.json configs[4], the one the metric is quoted on): aggregation microbench, k=3 objectives x P=1e8
parameters per GPU, aggregator `upgrad`, synthetic Jacobian (SURVEY 8d recipe).  One "step" = one pass of the hot path
over one resident Jacobian = ONE fused launch per GPU (csrc/aggregate.cu): Gramian pass -> (N > 1: k x k exchange over
NVLink peer memory inside the kernel) -> solve -> recombination pass + write-back.  metric = aggregation GB/s =
algorithmic bytes 4*P*(2k+1) per step (SURVEY 8d) / time, whole job over all N GPUs.  `--scaling weak` (default): P per
GPU fixed; `--scaling strong`: --P is the GLOBAL column count, split over the GPUs.  The timed region is a CUDA graph of
the K steps, entered through a device-side barrier over the peer flags (N > 1), timed with CUDA events, max over ranks.

Prints ONE compact JSON line (rank 0, < 4 KB); the per-leg evidence (quantizer shapes, train steps, optimizer, torch
context arms) goes to bench_detail_n<N>.json in --detail-dir (default: a new temporary directory, so that the benchmark
runs from a read-only checkout).  DESIGN.md section 4 explains every key.  `--dump-outputs DIR` writes what the timed
aggregation call returned in its last step (see `dump_outputs`), so that two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "aggregation_GBps"
UNIT = "GB/s"
LOSSES = [0.34, 1e-3, 2.5e-4, 0.17, 2.0]
DUMP_GRADIENT_COLUMNS = 1 << 22                   # 16 MB of float32: the dump stays far below 64 MB at any P


def workload_name(k: int, P: int, agg: str, scaling: str) -> str:
    """Byte-identical in both arms (the driver compares the strings)."""
    per = "per GPU" if scaling == "weak" else "global, P-sharded over the GPUs"
    return f"aggregation microbench k={k} P={P} {per} agg={agg} (BASELINE.json configs[4])"


def algorithmic_bytes(k: int, P: int) -> dict:
    return {"gram": 4 * k * P, "recombine": 4 * k * P + 4 * P, "step": 4 * P * (2 * k + 1)}


def measured_peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d.get("bf16_tflops", 1590.0)), "source": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback B200_PROFILING.md"}


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` capture
    of this workload (profiles/r2_traffic.json, else r1), or None."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            v = json.load(open(os.path.join(ROOT, "profiles", name))).get(kernel)
            if v is not None:
                return v
        except Exception:
            pass
    return None


def synthetic_J_into(J: torch.Tensor, seed: int, chunk: int = 1 << 24) -> None:
    """SURVEY 8d tier A: row i = s_i (0.3 g0 + sqrt(0.91) g_i), s = logspace(0,-1,k); generated on J's device."""
    k, P = J.shape
    gen = torch.Generator(device=J.device).manual_seed(seed)
    s = torch.logspace(0, -1, k, device=J.device)
    for c0 in range(0, P, chunk):
        c = min(chunk, P - c0)
        g0 = torch.randn(c, generator=gen, device=J.device)
        rows = torch.randn(k, c, generator=gen, device=J.device)
        J[:, c0:c0 + c] = s[:, None] * (0.3 * g0[None, :] + 0.91 ** 0.5 * rows)


class ClockSampler:
    """Samples SM clock and throttle reasons DURING the timed region (pynvml, ~every 2 ms)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        self.thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.thread is not None:
            self.thread.join()

    def summary(self) -> dict:
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def bind_to_gpu_numa_node(index: int):
    """Multi-GPU runs: pin this rank's host threads to the CPUs NVML reports as local to its GPU (first-touch of the
    pinned e2e buffers on the GPU's own NUMA node).  Best effort."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = (os.cpu_count() + 63) // 64 + 4
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, word in enumerate(mask) for b in range(64) if (int(word) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------ CPU arms (oracle)
def cpu_reference_run(k: int, P: int, agg: str, steps: int, warmup: int, budget_s: float):
    """The reference's CPU implementation of the path (oracle port: `J @ J.T` -> solve -> `w @ J` with the reference's
    own float32 torch expressions), all host threads, on a bounded sample of the workload."""
    from oracle import aggregation as oa

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(1234)
    losses = torch.tensor([LOSSES[i % len(LOSSES)] for i in range(k)])

    def make(Ps):
        s = torch.logspace(0, -1, k)
        J = torch.empty(k, Ps)
        for c0 in range(0, Ps, 1 << 24):
            c = min(1 << 24, Ps - c0)
            J[:, c0:c0 + c] = s[:, None] * (0.3 * torch.randn(c, generator=g)[None] + 0.91 ** 0.5 * torch.randn(k, c, generator=g))
        return J

    Ps = min(P, 10_000_000)
    J = make(Ps)
    t0 = time.perf_counter()
    oa.aggregate_reference_fp32(agg, J, losses)
    per_col = (time.perf_counter() - t0) / Ps
    Ps_fit = int(budget_s / max(per_col * (steps + warmup), 1e-12))      # size the sample so that warmup+steps fit the budget
    Ps = max(1_000_000, min(P, Ps_fit))
    if Ps != J.shape[1]:
        J = make(Ps)
    for _ in range(warmup):
        oa.aggregate_reference_fp32(agg, J, losses)
    t0 = time.perf_counter()
    for _ in range(steps):
        oa.aggregate_reference_fp32(agg, J, losses)
    total = time.perf_counter() - t0
    gbps = algorithmic_bytes(k, Ps)["step"] * steps / total / 1e9
    return {"value": gbps, "ms_per_step": 1e3 * total / steps, "cores": cores, "P_sample": Ps,
            "sample": f"k={k} P={Ps} of {P} ({'full' if Ps == P else 'bounded'}), {steps} steps after {warmup} warm-up, "
                      f"torch CPU f32, {cores} threads"}


def cpu_vq_codes_per_s(n_batch: int = 256, hw: int = 16) -> float:
    """Reference quantizer forward (oracle = vq_vae.py:27-64 expressions) on the host, N = n_batch*hw*hw code vectors."""
    from oracle import vq as ov

    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(4321)
    E = 0.5 * torch.randn(512, 64, generator=g)
    z = 0.5 * torch.randn(n_batch, 64, hw, hw, generator=g)
    ov.quantize_forward(z, E)
    t0 = time.perf_counter()
    for _ in range(3):
        ov.quantize_forward(z, E)
    return n_batch * hw * hw * 3 / (time.perf_counter() - t0)


def cpu_vae_steps_per_s(budget_s: float = 12.0) -> float:
    """BASELINE configs[0] end to end on the host cores (SURVEY 8d): the reference-style train step (tools/vqvae_harness.py
    `reference_style_step`: per-parameter reshape + cat, `J @ J.T`, float64 QP on the host, `w @ J`, per-tensor clone,
    both hooks, torch Adam) on CPU tensors."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from vqvae_harness import reference_style_runner

    torch.set_num_threads(os.cpu_count() or 1)
    step = reference_style_runner("vae", torch.device("cpu"))
    step()
    t0 = time.perf_counter()
    n = 0
    while n < 3 or (time.perf_counter() - t0 < budget_s and n < 30):
        step()
        n += 1
    return n / (time.perf_counter() - t0)


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args.k, args.P, args.agg, args.steps, max(args.warmup, 1), budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(r["value"], 3), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(r["ms_per_step"], 3), "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.k, args.P, args.agg, args.scaling), "timed_on": "host CPU", "sample_P": r["P_sample"]},
        "cpu_baseline": {"value": round(r["value"], 3), "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": round(r["value"], 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ extra legs (detail file)
def run_vq(dev, peaks: dict) -> dict:
    """Quantizer leg (K=512, D=64): nearest-codebook search, whole forward, backward, per kernel group with CUDA events; L2
    flushed between iterations.  Keys are the row counts N."""
    import movae_b200
    from movae_b200 import quantizer as Q

    out = {}
    gen = torch.Generator(device=dev).manual_seed(4321)
    E = 0.5 * torch.randn(512, 64, generator=gen, device=dev)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)       # 256 MB > L2
    vq = movae_b200.VectorQuantizer(512, 64).to(dev)
    with torch.no_grad():
        vq.embedding.weight.copy_(E)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    for (B, H, W), iters in (((128, 8, 8), 10), ((256, 16, 16), 10), ((64, 64, 64), 10), ((256, 128, 128), 5)):
        N = B * H * W
        z = 0.5 * torch.randn(B, 64, H, W, generator=gen, device=dev)
        zz = z.clone().requires_grad_(True)
        go = torch.randn_like(z)
        t_search = t_fwd = t_bwd = 0.0
        for i in range(iters + 2):
            flush.fill_(float(i))
            a, b, c, d = ev(), ev(), ev(), ev()
            a.record()
            Q.code_indices(z, E, 0)
            b.record()
            q, commit, embed, idx = vq(zz)
            c.record()
            torch.autograd.backward([q, commit, embed], [go, torch.ones_like(commit), torch.ones_like(embed)])
            d.record()
            torch.cuda.synchronize()
            zz.grad = None
            vq.embedding.weight.grad = None
            if i >= 2:
                t_search += a.elapsed_time(b)
                t_fwd += b.elapsed_time(c)
                t_bwd += c.elapsed_time(d)
        t_search, t_fwd, t_bwd = t_search / iters, t_fwd / iters, t_bwd / iters
        tf = N * 65536 / (t_search * 1e-3) / 1e12
        rec = {"search_ms": round(t_search, 4), "codes_per_s": round(N / (t_search * 1e-3), 1), "tflops_algorithmic": round(tf, 1),
               "frac_algorithmic": round(tf / peaks["bf16_tflops"], 4), "frac_executed": round(tf * 15.0 / 4.0 / peaks["bf16_tflops"], 4),
               "rechecked_rows_frac": round(Q.rechecked_rows(dev) / N, 5), "forward_ms": round(t_fwd, 4), "backward_ms": round(t_bwd, 4),
               "forward_GBps_776B_per_code": round(N * 776 / (t_fwd * 1e-3) / 1e9, 1),
               "backward_GBps_776B_per_code": round(N * 776 / (t_bwd * 1e-3) / 1e9, 1)}
        if N <= 262144:
            # the BASELINE shapes are launch-bound when driven eagerly from Python: the same forward + backward replayed
            # from a CUDA graph (how the train-step harness runs them) is the GPU time of the quantizer kernels themselves
            one = torch.ones((), device=dev)
            zg = z.clone().requires_grad_(True)
            vqg = movae_b200.VectorQuantizer(512, 64).to(dev)
            with torch.no_grad():
                vqg.embedding.weight.copy_(E)

            def fwd_bwd():
                q_, c_, e_, _ = vqg(zg)
                return torch.autograd.grad([q_, c_, e_], [zg, vqg.embedding.weight], grad_outputs=[go, one, one])

            def search_only():
                return Q.code_indices(z, E, 0)
            def search_x20():     # 20 searches inside ONE graph: kernel time without the per-replay launch latency
                return [Q.code_indices(z, E, 0) for _ in range(20)]
            for name, fn, per in (("fwd_bwd_graph_ms", fwd_bwd, 1), ("search_one_per_replay_ms", search_only, 1),
                                  ("search_graph_ms", search_x20, 20)):
                gstep = movae_b200.GraphedStep(fn, warmup=2)
                for _ in range(3):
                    gstep()
                reps = 20 if per == 1 else 5
                a, b = ev(), ev()
                a.record()
                for _ in range(reps):
                    gstep()
                b.record()
                torch.cuda.synchronize()
                rec[name] = round(a.elapsed_time(b) / (reps * per), 4)
                del gstep
            del zg, vqg

            def torch_fwd():      # context: the reference's torch expressions (vq_vae.py:28-47) on this GPU
                lat = z.permute(0, 2, 3, 1).contiguous().view(-1, 64)
                dist = torch.sum(lat ** 2, dim=1, keepdim=True) + torch.sum(E ** 2, dim=1) - 2 * torch.matmul(lat, E.t())
                inds = torch.argmin(dist, dim=1).unsqueeze(1)
                onehot = torch.zeros(inds.size(0), 512, device=dev)
                onehot.scatter_(1, inds, 1)
                return torch.matmul(onehot, E), inds
            for _ in range(2):
                torch_fwd()
            a, b = ev(), ev()
            a.record()
            for _ in range(5):
                torch_fwd()
            b.record()
            torch.cuda.synchronize()
            rec["torch_reference_expressions_forward_ms"] = round(a.elapsed_time(b) / 5, 4)
        out[f"N{N}"] = rec
        del z, zz, go
    # bulk code extraction (SURVEY 8f rank 3): 8 batches of N = 262,144 rows, best of 3 with a warmed extractor
    zb = [0.5 * torch.randn(64, 64, 64, 64, generator=gen, device=dev) for _ in range(2)]
    ex = movae_b200.CodeExtractor(vq)
    best, best_ref, codes = 1e9, 1e9, None
    for rep in range(4):
        ex.reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(8):
            ex.push(zb[i % 2])
        codes = ex.finish()
        dt = time.perf_counter() - t0
        if rep > 0:
            best = min(best, dt)
    for rep in range(3):      # the reference's way on the same GPU: int64 indices, synchronous .cpu() per batch
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        for i in range(8):
            Q.code_indices(zb[i % 2], E, 0).cpu()
        best_ref = min(best_ref, time.perf_counter() - t1)
    out["code_extraction"] = {"rows": int(codes.numel()), "batches": 8, "code_dtype": str(codes.dtype), "best_of": 3,
                              "codes_per_s_e2e": round(codes.numel() / best, 1),
                              "same_search_int64_sync_cpu_per_batch_codes_per_s": round(codes.numel() / best_ref, 1),
                              "usage_percent": round(ex.usage_percentage(), 2)}
    return out


def run_torch_gpu_context(J: torch.Tensor, w: torch.Tensor, flat_grad: torch.Tensor, nbytes: dict, iters: int = 3) -> dict:
    """Context only: the reference's own torch expressions for the two streaming passes on the SAME B200 -- `J @ J.T`
    and `weights @ J` + the `.grad` copy, i.e. cuBLAS with M = N = k."""
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    for _ in range(2):
        G = J @ J.T
        flat_grad.copy_(w @ J)
    t_g = t_r = 0.0
    for _ in range(iters):
        a, b, c = ev(), ev(), ev()
        a.record()
        G = J @ J.T                                   # noqa: F841
        b.record()
        flat_grad.copy_(w @ J)
        c.record()
        torch.cuda.synchronize()
        t_g += a.elapsed_time(b)
        t_r += b.elapsed_time(c)
    t_g, t_r = t_g / iters, t_r / iters
    return {"gram_ms": round(t_g, 4), "gram_GBps": round(nbytes["gram"] / (t_g * 1e-3) / 1e9, 1),
            "recombine_ms": round(t_r, 4), "recombine_GBps": round(nbytes["recombine"] / (t_r * 1e-3) / 1e9, 1)}


def run_optim(dev, peaks: dict, n: int = 100_000_000, iters: int = 20) -> dict:
    """K7 leg (SURVEY 8f rank 4): fused optimizer step over flat float32 buffers of n parameters."""
    import movae_b200

    out = {}
    p = torch.nn.Parameter(torch.randn(n, device=dev))
    for name, ctor, bpp in (("adam", lambda: movae_b200.Adam([p], lr=1e-4), 28),
                            ("adam+clip_grad_norm", lambda: movae_b200.Adam([p], lr=1e-4, max_grad_norm=1.0), 32),
                            ("sgd_momentum", lambda: movae_b200.SGD([p], lr=1e-4, momentum=0.9), 20)):
        if getattr(p, "_movae_flat", None) is not None:
            del p._movae_flat
        opt = ctor()
        p.grad = None
        opt.flat.adopt([p], [torch.randn(n, device=dev)])
        for _ in range(3):
            opt.step()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            opt.step()
        b.record()
        torch.cuda.synchronize(dev)
        ms = a.elapsed_time(b) / iters
        gbps = n * bpp / (ms * 1e-3) / 1e9
        out[name] = {"ms": round(ms, 4), "algorithmic_bytes_per_param": bpp, "GBps": round(gbps, 1),
                     "frac_of_hbm_peak": round(gbps / peaks["hbm_gbs"], 4)}
        del opt
    out["n_params"] = n
    return out


# ------------------------------------------------------------------------------------------------ the aggregation legs
class FusedLeg:
    """K steps of the fused aggregation over `windows` (a rotation of disjoint column windows of one big resident Jacobian:
    with more than one window every step streams memory no earlier step of the last 126 MB touched, so small-P numbers
    are cold-L2 numbers) captured into ONE CUDA graph; `run()` replays it between CUDA events."""

    def __init__(self, J_windows, out_windows, agg, exchange, steps: int):
        from movae_b200 import ops

        self.ops, self.exchange, self.steps = ops, exchange, steps
        self.dev = J_windows[0].device
        self.k = J_windows[0].shape[0]
        wt = agg.weighting
        if hasattr(agg, "_ensure_coef"):
            agg._ensure_coef(self.dev)
        wt.prepare_step(self.dev)
        self.spec, self.vec, self.aux = wt.solve_spec(self.k)
        self.Jw, self.ow = J_windows, out_windows
        self.last = None
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            for i in range(2):
                self._step(i)
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.ws = ops.current_workspace(self.dev, self.k)      # the capturing stream's workspace: holds the phase stamps
            for i in range(steps):
                self._step(i)

    def phase_times(self):
        """(Gramian pass, combine + exchange + solve, recombination pass) in ms of the LAST launch of the last replay."""
        torch.cuda.synchronize(self.dev)
        return self.ops.aggregate_phase_times(self.ws)

    def solve_breakdown_us(self) -> dict:
        """The solve phase of the last launch in its pieces (us): partial combine, k x k exchange, the solve itself."""
        torch.cuda.synchronize(self.dev)
        t0, t1, t2, t3, t4, t5 = self.ops.aggregate_stamps(self.ws)
        return {"combine_us": round((t4 - t1) * 1e-3, 1), "exchange_us": round((t5 - t4) * 1e-3, 1), "solve_only_us": round((t2 - t5) * 1e-3, 1)}

    def _step(self, i: int):
        n = len(self.Jw)
        self.last = self.ops.aggregate(self.Jw[i % n], self.spec, self.vec, self.aux, out=self.ow[i % n], exchange=self.exchange)

    def run(self, reps: int = 1) -> float:
        """ms per step (this rank), device-timed; every rep enters through the device-side barrier when N > 1."""
        best = 1e30
        for _ in range(reps):
            if self.exchange is not None:
                self.exchange.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            self.graph.replay()
            b.record()
            torch.cuda.synchronize(self.dev)
            best = min(best, a.elapsed_time(b) / self.steps)
        return best


def dump_outputs(path: str, w: torch.Tensor, diag: torch.Tensor, G: torch.Tensor, grad: torch.Tensor) -> None:
    """Writes what `ops.aggregate` returned to its caller as path/<name>.npy: weights.npy (float32 [k], [2k] for COMFORT),
    diag.npy (float64 [8]), gramian.npy (float64 [k, k]) and gradient.npy (float32).  A gradient longer than
    DUMP_GRADIENT_COLUMNS columns is sampled: the columns are torch.randint(P, (DUMP_GRADIENT_COLUMNS,)) drawn from a CPU
    generator seeded with 0, sorted, so the same P always gives the same columns."""
    P = grad.numel()
    if P > DUMP_GRADIENT_COLUMNS:
        cols = torch.randint(P, (DUMP_GRADIENT_COLUMNS,), generator=torch.Generator().manual_seed(0)).sort().values
        grad = grad[cols.to(grad.device)]
    os.makedirs(path, exist_ok=True)
    import numpy as np

    for name, t in (("weights", w), ("diag", diag), ("gramian", G), ("gradient", grad)):
        np.save(os.path.join(path, f"{name}.npy"), t.cpu().numpy())


def max_over_ranks(x: float, dev, world: int) -> float:
    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_movae(args) -> None:
    import torch.distributed as dist

    import movae_b200
    from movae_b200 import ops
    from movae_b200 import parallel as par

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (movae_b200 has no CPU fallback)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local)          # pinned e2e buffers first-touched on the GPU's own NUMA node
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")     # the DP leg captures NCCL collectives into a graph
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    k, K, W = args.k, args.steps, max(args.warmup, 3)
    strong = args.scaling == "strong"
    P_global = args.P if strong else world * args.P
    lo, hi = par.shard_columns(args.P, rank, world) if strong else (0, args.P)
    P = hi - lo                                              # this rank's columns
    P_alloc = max(P, 0 if strong else args.P)
    ld = (P_alloc + 31) // 32 * 32                           # rows start on 128-byte lines
    Jbuf = torch.empty((k, ld), dtype=torch.float32, device=dev)
    J = Jbuf[:, :P]
    synthetic_J_into(J, 1234 + rank)
    losses = torch.tensor([LOSSES[i % len(LOSSES)] for i in range(k)], device=dev)
    agg = movae_b200.make_aggregator(args.agg) if args.agg != "sum" else movae_b200.Sum()
    if isinstance(agg, movae_b200.MGDA) or hasattr(agg, "set_losses"):
        agg.set_losses(losses)
    flat_grad = torch.empty(ld, dtype=torch.float32, device=dev)[:P]
    nbytes = algorithmic_bytes(k, P)
    exchange = par.install_p2p_gramian_exchange(agg, dev) if world > 1 else None
    peaks = measured_peaks()

    # ---- parity gate before timing (torch float64 on a slice; N > 1: the exchanged Gramian against a NCCL all_reduce) ----
    leg = FusedLeg([J], [flat_grad], agg, exchange, K)
    w, diag, G_sum, _ = leg.last                             # the tensors the captured launches write
    leg.run()
    sl = min(P, 4_000_000)
    G_loc = ops.gram(J)
    G_ref = G_loc.clone()
    if world > 1:
        dist.all_reduce(G_ref)
    ref_sl = J[:, :sl].double() @ J[:, :sl].double().T
    if not torch.allclose(ops.gram(J[:, :sl]), ref_sl, rtol=1e-5, atol=1e-6):
        raise RuntimeError("bench parity gate failed: Gramian deviates from the float64 reference")
    g_rel = float(((G_sum - G_ref).abs().max() / G_ref.abs().max()).item())
    # the two Gramians come from different span decompositions (different float32 chain boundaries): equal to ~1e-11, while
    # a wrong exchange (a missing or doubled rank partial) is off by O(1 / N)
    if g_rel > 1e-9:
        raise RuntimeError(f"bench parity gate failed: exchanged / fused Gramian deviates from the reduced K1 Gramian ({g_rel:.3e})")
    w_sep = agg.weighting.from_gramian(G_ref)[:k]            # K2 alone on the reduced Gramian
    w_dev = float((w[:k] - w_sep).abs().max().item())
    ref_g = (w[:k].double() @ J[:, :sl].double()).float()
    if not torch.allclose(flat_grad[:sl], ref_g, rtol=1e-5, atol=1e-6):
        raise RuntimeError("bench parity gate failed: aggregated gradient deviates from the float64 reference")
    status = float(diag[4].item())
    if w_dev > 1e-6 or status != 0.0 or not par.check_replicated(w):
        raise RuntimeError(f"bench parity gate failed: weights (dev {w_dev:.3e}, status {status}, replicated {par.check_replicated(w)})")
    g_max_rel = float(((flat_grad[:sl] - ref_g).abs().max() / ref_g.abs().max()).item())
    parity = {"G_fused_vs_allreduce_rel": g_rel, "w_replicated_bitwise": True, "w_vs_separate_solve_max_abs": w_dev,
              "grad_vs_fp64_max_rel": g_max_rel, "status": int(status)}

    # ---- headline: W warm-up steps, then K steps (one graph) between events, max over ranks ----
    for _ in range((W + K - 1) // K):
        leg.run()
    barrier()
    with ClockSampler(local) as clocks:
        ms_step = leg.run()
        t_g, t_s, t_r = leg.phase_times()                     # the last launch's own globaltimer stamps
        brk = leg.solve_breakdown_us()
        ms2 = leg.run(reps=2)                                # the sampler needs more than one replay to see the load
        barrier()
    ms_step = max_over_ranks(ms_step, dev, world)
    ms_best = max_over_ranks(min(ms_step, ms2), dev, world)
    value = 4.0 * P_global * (2 * k + 1) / (ms_step * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, w, diag, G_sum, flat_grad)     # now: the legs below write into flat_grad again

    # ---- small / sharded sizes on the same Jacobian (cold L2 through window rotation) ----
    def windows_leg(P_win: int, label: str) -> dict:
        n_win = max(1, min(8, P // P_win))
        if n_win * P_win * 4 * (k + 1) < 300e6 and n_win < 8:
            return {}
        Pw = P_win // 32 * 32
        Jw = [Jbuf[:, i * Pw:i * Pw + P_win] for i in range(n_win)]
        ow = [flat_grad[i * Pw:i * Pw + P_win] for i in range(n_win)]
        lg = FusedLeg(Jw, ow, agg, exchange, max(K, 4 * n_win))
        lg.run()
        ms = max_over_ranks(lg.run(reps=3), dev, world)
        tg, ts, tr = lg.phase_times()
        b = algorithmic_bytes(k, P_win)
        return {f"{label}_ms_per_step": round(ms, 4), f"{label}_frac": round(b["step"] / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                f"{label}_gram_pass_frac": round(b["gram"] / (tg * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                f"{label}_recombine_pass_frac": round(b["recombine"] / (tr * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                f"{label}_solve_us": round(ts * 1e3, 1), f"{label}_windows": n_win}

    small = {}
    strong_block = None
    if not strong and P >= 80_000_000:
        if world == 1:
            small = windows_leg(10_000_000, "P1e7")
        else:
            # strong scaling of a FIXED global P = 1e8 (what configs[4] names): every rank streams P / N columns per step
            Ps = 100_000_000 // world // 32 * 32
            r = windows_leg(Ps, "strong")
            if r:
                gb = 4.0 * Ps * world * (2 * k + 1) / (r["strong_ms_per_step"] * 1e-3) / 1e9
                strong_block = {"global_P": Ps * world, "columns_per_gpu": Ps, "ms_per_step": r["strong_ms_per_step"],
                                "GBps_whole_job": round(gb, 1), "frac_of_N_x_hbm_peak": r["strong_frac"],
                                "gram_pass_frac": r["strong_gram_pass_frac"], "recombine_pass_frac": r["strong_recombine_pass_frac"],
                                "solve_plus_exchange_us": r["strong_solve_us"], "cold_l2_windows": r["strong_windows"]}

    # ---- e2e: HOST buffers through the C-ABI host pipeline, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        h_J = torch.empty((k, P), dtype=torch.float32, pin_memory=True)
        h_J.copy_(J)
        h_outs = [torch.empty(P, dtype=torch.float32, pin_memory=True) for _ in range(2)]
        plan = movae_b200.HostAggregationPlan(k, P, dev, depth=2)
        reducer = par.gramian_allreduce() if world > 1 else None
        e_steps = args.e2e_steps if args.e2e_steps > 0 else K
        for i in range(2):
            plan.run_async(h_J, agg, h_outs[i % 2], reducer)
        plan.wait()
        barrier()
        t0 = time.perf_counter()
        for i in range(e_steps):
            # every step: H2D of its Jacobian from pinned host memory, the three kernels per column chunk, D2H of its result;
            # consecutive steps are pipelined over two sets of device buffers (step i's D2H overlaps step i+1's H2D)
            plan.run_async(h_J, agg, h_outs[i % 2], reducer)
        plan.wait()                                  # every result is in host memory
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - t0, dev, world)
        torch.cuda.synchronize()
        leg.run()                                    # flat_grad as the resident path writes it
        h_out = h_outs[(e_steps - 1) % 2]
        e2e = {"value": round(4.0 * P_global * (2 * k + 1) * e_steps / e2e_s / 1e9, 2), "unit": UNIT, "h2d_bytes_per_step": 4 * k * P,
               "d2h_bytes_per_step": 4 * P, "steps": e_steps, "api": "HostAggregationPlan.run_async + wait, pinned host buffers, 2 steps in flight",
               "max_abs_dev_vs_resident": float((h_out.to(dev) - flat_grad).abs().max())}
        del h_J, h_out, h_outs, plan

    # ---- extra legs -> detail file; a few scalars of them -> the line ----
    detail, flat_roof, flat_cpu = {}, {}, {}
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    if not args.quick:
        if world > 1:
            from movae_b200 import quantizer as Q
            from vqvae_harness import time_dp_train_steps

            gen = torch.Generator(device=dev).manual_seed(4321 + rank)
            E = 0.5 * torch.randn(512, 64, generator=torch.Generator(device=dev).manual_seed(4321), device=dev)   # replicated codebook
            zq = 0.5 * torch.randn(256, 64, 128, 128, generator=gen, device=dev)                                  # this rank's rows
            for _ in range(3):
                Q.code_indices(zq, E, 0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            a.record()
            for _ in range(10):
                Q.code_indices(zq, E, 0)
            b.record()
            barrier()
            tq = max_over_ranks(a.elapsed_time(b) / 10, dev, world)
            n_local = zq.shape[0] * zq.shape[2] * zq.shape[3]
            detail["vq_sharded"] = {"rows_per_gpu": n_local, "search_ms_max_over_ranks": round(tq, 4),
                                    "codes_per_s_whole_job": round(world * n_local / (tq * 1e-3), 1)}
            flat_roof["vq_sharded_codes_per_s"] = detail["vq_sharded"]["codes_per_s_whole_job"]
            del zq
            detail["train_step_data_parallel"] = time_dp_train_steps(dev, rank, world)
            flat_roof["dp_vqvae_steps_per_s_graph"] = detail["train_step_data_parallel"]["graph"]["steps_per_s"]
        elif rank == 0:
            from vqvae_harness import (time_ggvqvae_train_steps, time_train_steps, time_vae_train_steps, time_vqvae2_train_steps)

            w_now = w[:k].clone()
            detail["torch_gpu_context"] = run_torch_gpu_context(J, w_now, flat_grad, nbytes)
            leg.run()
            detail["optim"] = run_optim(dev, peaks)
            detail["vq"] = run_vq(dev, peaks)
            for n in ("N262144", "N4194304"):
                v = detail["vq"][n]
                flat_roof[f"vq_{n}_codes_per_s"] = v["codes_per_s"]
                flat_roof[f"vq_{n}_frac_algorithmic"] = v["frac_algorithmic"]
            flat_roof["vq_N4194304_frac_executed"] = detail["vq"]["N4194304"]["frac_executed"]
            sustained = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops_sustained") if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else None
            if sustained:      # executed flops against what cuBLAS sustains on this part (power-limited), not the burst peak
                flat_roof["vq_N4194304_frac_executed_of_sustained_peak"] = round(detail["vq"]["N4194304"]["tflops_algorithmic"] * 3.75 / float(sustained), 4)
            flat_roof["vq_algorithmic_ceiling_of_bf16x3_split"] = round(4.0 / 15.0, 4)
            flat_roof["vq_search_us_N8192_N65536_N262144"] = [round(1e3 * detail["vq"][n].get("search_graph_ms", detail["vq"][n]["search_ms"]), 1)
                                                             for n in ("N8192", "N65536", "N262144")]
            for key, fn in (("vqvae", time_train_steps), ("vae", time_vae_train_steps), ("ggvqvae", time_ggvqvae_train_steps),
                            ("vqvae2", time_vqvae2_train_steps)):
                r = fn(dev)
                detail[f"train_step_{key}"] = r
                flat_roof[f"steps_per_s_{key}"] = r["movae_graph_e2e"]["steps_per_s"]
                if "reference_style" in r:
                    flat_roof[f"steps_per_s_{key}_reference_style_gpu"] = r["reference_style"]["steps_per_s"]

    if rank == 0:
        frac = nbytes["step"] / (ms_step * 1e-3) / 1e9 / peaks["hbm_gbs"]
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(k, args.P, args.agg, args.scaling), "global_P": P_global, "columns_this_gpu": P,
                       "sharding": (f"P-sharded x{world}, k*k float64 exchange over NVLink peer memory inside the kernel" if world > 1 else "single GPU"),
                       "l2": f"inputs larger than L2 ({(nbytes['gram'] + 4 * P) / 1e6:.0f} MB per GPU vs 126 MB), no flush",
                       "timed": f"one CUDA graph of {K} fused launches, CUDA events, max over ranks" + (", device-side start barrier" if world > 1 else "")},
            "roofline": {"bound": "hbm", "kernel": "aggregate_kernel", "achieved": round(nbytes["step"] / (ms_step * 1e-3) / 1e9, 1),
                         "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(frac, 4), "traffic": ncu_traffic("aggregate_kernel"),
                         "peak_source": peaks["source"], "frac_of_nominal_8000": round(frac * peaks["hbm_gbs"] / 8000.0, 4),
                         "algorithmic_bytes_per_launch": nbytes["step"],
                         "gram_pass_ms": round(t_g, 4), "gram_pass_frac": round(nbytes["gram"] / (t_g * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                         "solve_us": round(t_s * 1e3, 1), **brk,
                         "recombine_pass_ms": round(t_r, 4), "recombine_pass_frac": round(nbytes["recombine"] / (t_r * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                         "best_ms_per_step": round(ms_best, 4), **small, **flat_roof},
            "gpu_launches": K,
            "clocks": clocks.summary(),
            "multi_gpu_parity" if world > 1 else "parity": parity,
        }
        if e2e is not None:
            line["e2e"] = e2e
        if world > 1:       # the same facts as flat scalars / one string inside keys every consumer of the line keeps
            line["config"]["multi_gpu_parity"] = (f"G fused-exchange vs NCCL all_reduce rel {parity['G_fused_vs_allreduce_rel']:.1e}; w bitwise replicated; "
                                                  f"w vs K2-on-reduced-G {parity['w_vs_separate_solve_max_abs']:.1e}; grad vs fp64 rel {parity['grad_vs_fp64_max_rel']:.1e}")
        if strong_block is not None:
            line["strong"] = strong_block
            line["roofline"].update({"strong_global_P": strong_block["global_P"], "strong_ms_per_step": strong_block["ms_per_step"],
                                     "strong_GBps_whole_job": strong_block["GBps_whole_job"],
                                     "strong_frac_of_N_x_hbm_peak": strong_block["frac_of_N_x_hbm_peak"]})
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)        # the CPU baseline gets every host core again
            r = cpu_reference_run(k, P, args.agg, steps=3, warmup=1, budget_s=15.0)
            cb = {"value": round(r["value"], 3), "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]}
            if not args.quick:
                cb["vq_codes_per_s_N65536"] = round(cpu_vq_codes_per_s(), 1)
                cb["vae_configs0_steps_per_s"] = round(cpu_vae_steps_per_s(), 3)
            line["cpu_baseline"] = cb
        if detail:
            detail_dir = args.detail_dir or tempfile.mkdtemp(prefix="movae_bench_")
            os.makedirs(detail_dir, exist_ok=True)
            path = os.path.abspath(os.path.join(detail_dir, f"bench_detail_n{world}.json"))
            with open(path, "w") as f:
                json.dump({"line": line, "detail": detail}, f, indent=1)
            line["detail_file"] = path
        print(json.dumps(line), flush=True)
    if world > 1:
        # CUDA graphs that captured NCCL kernels may still be alive: tearing the communicator down under them can block
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="movae", choices=["movae", "reference"])
    ap.add_argument("--k", type=int, default=3)
    ap.add_argument("--P", type=int, default=100_000_000)
    ap.add_argument("--agg", default="upgrad")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer leg (0 = --steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline + roofline + e2e only: skip the quantizer / train-step / optimizer legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's weights, diagnostics, Gramian and "
                                                          "(sampled) gradient to DIR/<name>.npy (movae arm, rank 0)")
    ap.add_argument("--detail-dir", metavar="DIR", help="where bench_detail_n<N>.json goes (default: a new temporary directory)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs needs --impl movae: the reference arm times the CPU oracle on a sample of the columns")
    sys.dont_write_bytecode = True            # the checkout may be read-only: no __pycache__ beside the sources
    if args.impl == "reference":
        run_reference(args)
    else:
        run_movae(args)


if __name__ == "__main__":
    main()
