"""Timing of VectorQuantizerEMA's codebook update on one GPU (K = 512, D = 64).

    python tools/vq_ema_bench.py [--sizes 8192,65536,262144,4194304] [--rounds 5] [--out FILE]

For each N it reports, in one markdown table:
  - the update alone (statistics + apply, `VectorQuantizerEMA._update`): 20 updates captured in one CUDA graph, timed
    with CUDA events after warm-up.  The latents rotate over enough distinct buffers that every graph replay reads more
    than twice the 126 MB L2 (at N = 4,194,304 one 1.07 GB buffer already does);
  - beside it, K6b plus vq_dE_reduce_kernel (the codebook-gradient half of VectorQuantizer's backward, which reads the
    same bytes), timed the same way;
  - GB/s of the update on algorithmic bytes N (4 D + 8) (latents and indices) plus the state bytes 8 K + 20 K D
    (cluster_size read and written; embed_avg read and written; the codebook read, copied and written), against the
    measured copy peak of 6546.6 GB/s;
  - the whole forward + backward of VectorQuantizer and of VectorQuantizerEMA (training mode), eager, CUDA events,
    alternating the two classes round by round; the median over rounds.
The GPU name and power limit are read in the same run and printed above the table.
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import movae_b200  # noqa: E402
from movae_b200 import _lib as L  # noqa: E402

K, D = 512, 64
COPY_PEAK_GBPS = 6546.6
L2_BYTES = 126 * 2 ** 20
GRAPH_LEN = 20


def gpu_header() -> str:
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unavailable"
    return f"GPU: {name}; power limit, max SM clock: {q}; torch {torch.__version__}"


def shape_for(N: int):
    """[B, 64, H, W] with H * W = 64 * 64 (H * W % 32 == 0: the TMA statistics kernel) or fewer rows when N is small."""
    hw = 4096 if N >= 4096 else N
    return N // hw, D, hw // 64 if hw >= 64 else 1, 64 if hw >= 64 else hw


def time_graph(fns, reps: int) -> float:
    """ms per call of the callables in `fns` (each one step), captured GRAPH_LEN at a time; graphs replayed round robin."""
    graphs = []
    side = torch.cuda.Stream()             # warm-up and capture on one stream: its workspaces exist before the capture
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for f in fns:
            f()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for g0 in range(0, len(fns), GRAPH_LEN):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for i in range(GRAPH_LEN):
                fns[(g0 + i) % len(fns)]()
        graphs.append(g)
    for g in graphs:                                      # warm-up replays
        g.replay()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for r in range(reps):
        for g in graphs:
            g.replay()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / (reps * len(graphs) * GRAPH_LEN)


def bench_size(N: int, rounds: int, dev) -> dict:
    B, _, H, W = shape_for(N)
    gen = torch.Generator(device=dev).manual_seed(N)
    z_bytes = N * (4 * D + 8)
    n_buf = max(1, min(128, -(-2 * L2_BYTES // z_bytes)))
    zs = [0.5 * torch.randn(B, D, H, W, generator=gen, device=dev) for _ in range(n_buf)]
    ema = movae_b200.VectorQuantizerEMA(K, D).to(dev)
    with torch.no_grad():
        ema.embedding.weight.copy_(0.5 * torch.randn(K, D, generator=gen, device=dev))
        ema.embed_avg.copy_(ema.embedding.weight * 20.0)
        ema.cluster_size.fill_(20.0)
    idxs = [ema.get_code_indices(z) for z in zs]
    n_fns = max(GRAPH_LEN, n_buf)
    upd = [lambda i=i: ema._update(zs[i % n_buf], idxs[i % n_buf]) for i in range(n_fns)]
    t_upd = time_graph(upd, reps=max(3, 200 // n_fns))

    # K6b + vq_dE_reduce_kernel: VectorQuantizer's codebook-gradient pass over the same latents and indices
    E = ema.embedding.weight.detach().clone()
    dE = torch.zeros_like(E)
    g_embed = torch.ones(1, device=dev)
    need = L.lib().movae_vq_backward_workspace_bytes(N, K, D)
    scratch = torch.empty(need, dtype=torch.uint8, device=dev)

    def k6b(i):
        z, idx = zs[i % n_buf], idxs[i % n_buf]
        L.check(L.lib().movae_vq_backward_f32(0, 0, L.ptr(g_embed), L.ptr(z), B, D, H * W, L.ptr(E), K, L.ptr(idx), 0, L.ptr(dE),
                                              L.ptr(scratch), need, L.stream_of(z)), "vq_backward_f32")
    t_k6b = time_graph([lambda i=i: k6b(i) for i in range(n_fns)], reps=max(3, 200 // n_fns))

    # whole forward + backward, eager, the two classes alternating
    ref = movae_b200.VectorQuantizer(K, D).to(dev)
    with torch.no_grad():
        ref.embedding.weight.copy_(E)
    r = torch.randn(B, D, H, W, generator=gen, device=dev)
    zin = zs[0].clone().requires_grad_(True)

    def fwd_bwd(vq):
        zin.grad = None
        vq.embedding.weight.grad = None
        q, c, e, _ = vq(zin)
        (torch.sum(q * r) + 0.25 * c + e).backward()

    times = {"VectorQuantizer": [], "VectorQuantizerEMA": []}
    for vq in (ref, ema, ref, ema):                       # warm-up
        fwd_bwd(vq)
    iters = max(5, min(200, (1 << 24) // N))
    for _ in range(rounds):
        for name, vq in (("VectorQuantizer", ref), ("VectorQuantizerEMA", ema)):
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(iters):
                fwd_bwd(vq)
            e.record()
            torch.cuda.synchronize()
            times[name].append(s.elapsed_time(e) / iters)
    state_bytes = 8 * K + 20 * K * D
    gbps = (z_bytes + state_bytes) / (t_upd * 1e-3) / 1e9
    return {"N": N, "buffers": n_buf, "update_ms": t_upd, "k6b_reduce_ms": t_k6b, "GBps": gbps, "frac": gbps / COPY_PEAK_GBPS,
            "fb_vq_ms": statistics.median(times["VectorQuantizer"]), "fb_ema_ms": statistics.median(times["VectorQuantizerEMA"])}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--sizes", default="8192,65536,262144,4194304")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the markdown table to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("vq_ema_bench.py needs a CUDA device")
    dev = torch.device("cuda")
    lines = [gpu_header(), "",
             "| N | latent buffers | update ms (stats + apply) | K6b + dE reduce ms | update / K6b | update GB/s | of 6546.6 GB/s "
             "| fwd+bwd VectorQuantizer ms | fwd+bwd VectorQuantizerEMA ms |",
             "|---|---|---|---|---|---|---|---|---|"]
    for N in (int(s) for s in args.sizes.split(",")):
        r = bench_size(N, args.rounds, dev)
        lines.append(f"| {r['N']:,} | {r['buffers']} | {r['update_ms']:.4f} | {r['k6b_reduce_ms']:.4f} | "
                     f"{r['update_ms'] / r['k6b_reduce_ms']:.3f} | {r['GBps']:.1f} | {r['frac']:.3f} | {r['fb_vq_ms']:.4f} | "
                     f"{r['fb_ema_ms']:.4f} |")
        print(lines[-1], flush=True)
        torch.cuda.empty_cache()
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
