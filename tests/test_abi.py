"""CPU tests: the C-ABI library loads and exports every symbol include/movae_b200.h declares
(no compute calls -- there is no GPU here), and the product path refuses to run without CUDA."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "movae_b200.h")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(movae_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import movae_b200
    from movae_b200 import _lib

    assert os.path.exists(movae_b200.LIB_PATH), "run `python mo-vae_b200/build.py` (or __graft_entry__.build())"
    handle = ctypes.CDLL(movae_b200.LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 10
    for n in names:
        assert hasattr(handle, n), f"{n} declared in the header but not exported"
    assert set(names) == set(_lib.exported_symbols()), "ctypes binding out of sync with the header"
    assert movae_b200.lib().movae_abi_version() == _lib.ABI_VERSION


def test_workspace_query_is_host_only():
    import movae_b200

    lib = movae_b200.lib()
    assert lib.movae_gram_workspace_bytes(0) == 0
    assert lib.movae_gram_workspace_bytes(9) == 0
    assert lib.movae_gram_workspace_bytes(3) >= 256 + 6 * 8
    assert lib.movae_gram_workspace_bytes(8) > lib.movae_gram_workspace_bytes(3)


def test_fused_segment_launch_rejects_a_misaligned_workspace():
    import movae_b200
    from movae_b200 import _lib

    lib = movae_b200.lib()
    segs = _lib.JacSegments(n_segments=1, k=1)
    segs.n[0] = 4
    segs.rows[0][0] = 0x10000                                          # never dereferenced: validation fails first
    spec = _lib.SolveSpec(kind=_lib.SOLVE_CONSTANT)
    ws_bytes = lib.movae_gram_workspace_bytes(1)
    rc = lib.movae_aggregate_segments_f32(ctypes.byref(segs), ctypes.byref(spec), None, None, None, 0, 0x20000, None, None,
                                          0x30004, ws_bytes, None, None)
    assert rc == 4, lib.movae_last_error()                            # MOVAE_ERR_WORKSPACE
    assert b"8-byte aligned" in lib.movae_last_error()


def test_optimizer_and_extraction_host_side_contracts():
    import ctypes

    import movae_b200
    from movae_b200 import _lib

    lib = movae_b200.lib()
    assert lib.movae_optim_state_bytes() >= 12
    assert ctypes.sizeof(_lib.OptimSpec) == 8 + 6 * 8                   # mirrors movae_optim_spec: 2 int32 + 6 float64
    assert movae_b200.make_optimizer.__doc__ and "main.py:1169" in movae_b200.make_optimizer.__doc__
    with pytest.raises(ValueError):
        movae_b200.make_optimizer("lion", [torch.nn.Parameter(torch.zeros(1))], lr=0.1)
    with pytest.raises(RuntimeError, match="CUDA"):
        movae_b200.Adam([torch.nn.Parameter(torch.zeros(3))], lr=0.1)    # no CPU fallback
    with pytest.raises(RuntimeError):
        movae_b200.parallel.DataParallel(movae_b200.Sum())                # needs an initialised process group


def test_product_path_refuses_cpu_tensors():
    import movae_b200

    for agg in (movae_b200.UPGrad(), movae_b200.AlignedMTL(), movae_b200.MGDA("l2"), movae_b200.Sum()):
        with pytest.raises(RuntimeError, match="CUDA"):
            agg(torch.randn(3, 16))
        with pytest.raises(ValueError):
            agg(torch.randn(16))


def test_constructor_errors_match_reference():
    import movae_b200

    with pytest.raises(ValueError):            # mgda.py:97-101
        movae_b200.MGDA(norm_type="bogus")
    m = movae_b200.MGDA(norm_type="loss")
    with pytest.raises(ValueError):            # mgda.py:215-218
        m.set_losses(torch.ones(2, 2))
    with pytest.raises(ValueError):            # main.py:1245
        movae_b200.make_aggregator("nonsense")
    assert movae_b200.make_aggregator("sum") == "sum" and movae_b200.make_aggregator(None) is None
    assert isinstance(movae_b200.make_aggregator("mgda_lgn"), movae_b200.MGDA)
    assert isinstance(movae_b200.make_aggregator("amtl"), movae_b200.AlignedMTL)
    assert movae_b200.make_aggregator("mgda_gn").mgda_weighting.norm_type == "loss"


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "mo-vae_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{f} imports the oracle"
