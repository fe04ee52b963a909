"""Aggregation microbench grid of BASELINE.json configs[4] on one GPU: k in {2,3,8} x P in {1e7,1e8,1e9}, every aggregator
of north_star, each as ONE fused launch replayed from a CUDA graph of 10 (P = 1e7: rotating over 8 disjoint windows of a
bigger Jacobian so that every launch is cold in L2) -> markdown table (profiles/r2_agg_sweep.md).  The graph is captured and
replayed through GraphedStep, so aggregators with a per-step host draw (PCGrad, PNUPGrad) are timed with their draw.
    python tools/agg_sweep.py [--max-bytes 60e9] [--names upgrad,pcgrad,imtlg]"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import movae_b200  # noqa: E402
from movae_b200 import ops  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--max-bytes", type=float, default=60e9)
ap.add_argument("--names", default=None, help="comma-separated aggregator names for every (k, P); default: the north_star list")
a = ap.parse_args()
dev = torch.device("cuda")
peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
LOSSES = [0.34, 1e-3, 2.5e-4, 0.17, 2.0]
print(f"# r2: fused aggregation launch, k x P x aggregator (one B200; fractions of the measured HBM peak {peak:.0f} GB/s)\n")
print("| k | P | aggregator | ms per launch | GB/s algorithmic | fraction | Gramian pass | solve phase (us) | recombination pass |")
print("|---|---|---|---|---|---|---|---|---|")
for k in (2, 3, 8):
    for P in (10_000_000, 100_000_000, 1_000_000_000):
        n_win = 8 if P == 10_000_000 else 1
        Pa = P * n_win
        if 4.0 * (k + 1) * Pa > a.max_bytes:
            print(f"| {k} | {P:.0e} | (skipped: {4.0 * (k + 1) * Pa / 1e9:.0f} GB > --max-bytes) | | | | | | |")
            continue
        J = torch.empty((k, Pa), dtype=torch.float32, device=dev)
        gen = torch.Generator(device=dev).manual_seed(1234)
        s = torch.logspace(0, -1, k, device=dev)
        for c0 in range(0, Pa, 1 << 24):
            c = min(1 << 24, Pa - c0)
            g0 = torch.randn(c, generator=gen, device=dev)
            J[:, c0:c0 + c] = s[:, None] * (0.3 * g0[None] + 0.91 ** 0.5 * torch.randn(k, c, generator=gen, device=dev))
        out = torch.empty(Pa, dtype=torch.float32, device=dev)
        losses = torch.tensor([LOSSES[i % 5] for i in range(k)], device=dev)
        names = ("upgrad", "aligned_mtl", "aligned_mtl_median", "mgda_ln", "mgda_gn", "mgda_lgn", "jd_sum") if P < 1_000_000_000 else ("upgrad", "aligned_mtl")
        if a.names:
            names = tuple(a.names.split(","))
        for name in names:
            agg = movae_b200.make_aggregator(name)
            if isinstance(agg, movae_b200.MGDA):
                agg.set_losses(losses)
            Jw = [J[:, i * P:(i + 1) * P] for i in range(n_win)]
            ow = [out[i * P:(i + 1) * P] for i in range(n_win)]
            steps = 16 if n_win > 1 else 10
            agg.aggregate_into(Jw[0], ow[0])                     # eager once: per-step device state (PCGrad's table) exists
            captured = {}

            def run_steps():
                if torch.cuda.is_current_stream_capturing():
                    captured["ws"] = ops.current_workspace(J.device, k)     # the capturing stream's workspace holds the stamps
                for i in range(steps):
                    agg.aggregate_into(Jw[i % n_win], ow[i % n_win])
            graph = movae_b200.GraphedStep(run_steps, warmup=1)
            ws = captured["ws"]
            graph()
            best = 1e30
            for _ in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                graph()
                e1.record()
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1) / steps)
            tg, ts, tr = ops.aggregate_phase_times(ws)
            b1, b3 = 4.0 * k * P, 4.0 * (k + 1) * P
            print(f"| {k} | {P:.0e} | {name} | {best:.4f} | {(b1 + b3) / best / 1e6:.0f} | {(b1 + b3) / best / 1e6 / peak:.3f} | "
                  f"{b1 / tg / 1e6 / peak:.3f} | {ts * 1e3:.1f} | {b3 / tr / 1e6 / peak:.3f} |", flush=True)
            del graph
        del J, out
        torch.cuda.empty_cache()
