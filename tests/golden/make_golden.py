"""Generates the committed golden fixtures by executing the REFERENCE'S OWN files
(/root/reference/utils/torchmoo/{aligned_mtl,mgda}.py, /root/reference/models/vq_vae.py) behind
oracle/ref_shim.py.  Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

Outputs (small, committed): tests/golden/aggregation_golden.json, tests/golden/vq_golden.npz (read it through
`load_vq_golden`)
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
LOSSES = [0.34, 1e-3, 2.5e-4, 0.17, 2.0]   # SURVEY 8d: measured loss magnitudes


def synthetic_J(k: int, P: int, seed: int, decades: float = 1.0, zero_row: int | None = None) -> torch.Tensor:
    """SURVEY 8d recipe: row i = s_i (c g0 + sqrt(1-c^2) g_i), c = 0.3, s = logspace(0,-decades,k)."""
    g = torch.Generator().manual_seed(seed)
    g0 = torch.randn(P, generator=g)
    rows = torch.randn(k, P, generator=g)
    c = 0.3
    s = torch.logspace(0, -decades, k)
    J = s[:, None] * (c * g0[None, :] + (1 - c * c) ** 0.5 * rows)
    if zero_row is not None:
        J[zero_row] = 0
    return J.contiguous()


def losses_for(k: int) -> torch.Tensor:
    return torch.tensor([LOSSES[i % len(LOSSES)] for i in range(k)], dtype=torch.float32)


def main() -> None:
    torch.set_num_threads(1)
    amtl = ref_shim.load_reference_aligned_mtl()
    mgda = ref_shim.load_reference_mgda()
    vqmod = ref_shim.load_reference_vq()
    nup = ref_shim.load_reference_nupgrad()
    pnup = ref_shim.load_reference_pnupgrad()

    cases = []
    kat_J = torch.tensor([[-4.0, 1.0, 1.0], [6.0, 1.0, 1.0]])
    zero_J = torch.tensor([[-4.0, 1.0, 1.0], [0.0, 0.0, 0.0], [6.0, 1.0, 1.0]])
    mats = [("kat", kat_J, torch.tensor([0.5, 2.0])), ("kat_zero_row", zero_J, torch.tensor([0.5, 1.0, 2.0]))]
    for k in (2, 3, 4, 5, 8):
        mats.append((f"tierA_k{k}", synthetic_J(k, 4099, 1234 + k, 1.0), losses_for(k)))
    mats.append(("tierA_k3_zero_row", synthetic_J(3, 4099, 77, 1.0, zero_row=1), losses_for(3)))
    mats.append(("tierB_k3", synthetic_J(3, 4099, 78, 2.0), losses_for(3)))
    mats.append(("dup_rows_k3", torch.stack([kat_J[0], kat_J[0], kat_J[1]]), losses_for(3)))

    for tag, J, losses in mats:
        G = (J.double() @ J.double().T).float()      # arbiter Gramian (fp64-accumulated, rounded once)
        entry = {"tag": tag, "k": int(J.shape[0]), "G": G.tolist(), "losses": losses.tolist(), "out": {}}
        if J.shape[1] <= 8:
            entry["J"] = J.tolist()
        for mode in ("min", "median", "rmse"):
            W = amtl.AlignedMTLWeighting(None, scale_mode=mode)
            entry["out"][f"aligned_mtl:{mode}"] = {"w": W(G).tolist()}
        for norm in ("none", "l2", "loss", "loss+"):
            W = mgda.MGDAWeighting(norm_type=norm)
            W.set_losses(losses)
            w = W(G)
            entry["out"][f"mgda:{norm}"] = {
                "w": w.tolist(), "convergence_count": int(W.convergence_count), "gamma": float(W.gamma)}
        W = mgda.MGDAWeighting(norm_type="l2", stable=True, min_eigenvalue_eps=1e-3)
        entry["out"]["mgda:l2:stable1e-3"] = {"w": W(G).tolist(), "convergence_count": int(W.convergence_count),
                                              "gamma": float(W.gamma)}
        # NUPGrad / PNUPGrad: the reference's own normalisation + wrapper code; the QP behind project_weights is the
        # oracle's restatement of quadprog (torchjd is not installable), so these pin the NORMALISATION semantics
        entry["out"]["nupgrad"] = {"w": nup._NUPGradWrapper(nup.MeanWeighting(), norm_eps=1e-4, reg_eps=1e-4, solver="quadprog")(G).tolist()}
        for prob, key in ((1.0, "pnupgrad:l2"), (0.0, "pnupgrad:min_l2")):
            Wp = pnup._PNUPGradWrapper(pnup.MeanWeighting(), prob=prob, norm_eps=1e-4, reg_eps=1e-4, solver="quadprog")
            entry["out"][key] = {"w": Wp(G).tolist()}
        if "J" in entry:   # full aggregator call on the tiny matrices (docstring KATs mgda.py:57-86)
            for norm in ("none", "l2", "loss", "loss+"):
                A = mgda.MGDA(norm_type=norm)
                A.set_losses(losses)
                entry["out"][f"mgda:{norm}"]["g"] = A(J).tolist()
            for mode in ("min", "median", "rmse"):
                entry["out"][f"aligned_mtl:{mode}"]["g"] = amtl.AlignedMTL(scale_mode=mode)(J).tolist()
        cases.append(entry)

    with open(os.path.join(HERE, "aggregation_golden.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_golden.py", "torch": torch.__version__, "cases": cases}, f)

    # ---- quantizer: reference module on seeded inputs, incl. exact-tie codebook -------------
    out = {}
    for tag, seed, trained, dup in (("init", 0, False, False), ("trained", 1, True, False), ("dup", 2, True, True)):
        torch.manual_seed(seed)
        B, D, H, W, K = 4, 64, 8, 8, 512
        vq = vqmod.VectorQuantizer(K, D)
        if trained:
            vq.embedding.weight.data.copy_(0.5 * torch.randn(K, D))
        if dup:   # duplicated codebook rows -> exact ties -> first index must win
            vq.embedding.weight.data[256:] = vq.embedding.weight.data[:256]
        z = (0.5 * torch.randn(B, D, H, W)).requires_grad_(True)
        r = torch.randn(B, D, H, W)
        q, commit, embed, idx = vq(z)
        (torch.sum(q * r) + 0.7 * commit + 1.3 * embed).backward()
        out[f"{tag}_z"] = z.detach().numpy()
        out[f"{tag}_E"] = vq.embedding.weight.detach().numpy().copy()
        out[f"{tag}_r"] = r.numpy()
        out[f"{tag}_q"] = q.detach().numpy()
        out[f"{tag}_commit"] = np.float32(commit.item())
        out[f"{tag}_embed"] = np.float32(embed.item())
        out[f"{tag}_idx"] = idx.numpy()
        out[f"{tag}_dz"] = z.grad.numpy()
        out[f"{tag}_dE"] = vq.embedding.weight.grad.numpy()
        out[f"{tag}_usage"] = np.float64(vq.get_codebook_usage_percentage_from_indices(idx))
    np.savez_compressed(os.path.join(HERE, "vq_golden.npz"), **{key: v for key, v in out.items() if not key.endswith("_dz")})
    rebuilt = load_vq_golden()
    for key, v in out.items():
        assert np.array_equal(rebuilt[key], v) and rebuilt[key].dtype == v.dtype, f"{key} is not rebuilt bit for bit"
    print("wrote", os.listdir(HERE))


def load_vq_golden() -> dict:
    """tests/golden/vq_golden.npz as a dict.  Each tag's `dz` is left out of the file (it would take it over 1 MB) and
    rebuilt here: the gradient `r` through the straight-through output plus 0.7 x the commitment loss' gradient
    2 (z - E[idx]) / N, in float32.  main() checks that this equals the reference module's autograd bit for bit."""
    gold = dict(np.load(os.path.join(HERE, "vq_golden.npz")))
    for tag in ("init", "trained", "dup"):
        z, E, r = gold[f"{tag}_z"], gold[f"{tag}_E"], gold[f"{tag}_r"]
        B, D, H, W = z.shape
        e = E[gold[f"{tag}_idx"]].reshape(B, H, W, D).transpose(0, 3, 1, 2)
        gold[f"{tag}_dz"] = r + np.float32(0.7 * 2 / z.size) * (z - e)
    return gold


if __name__ == "__main__":
    main()
