"""CPU tests of the host-side layout logic of FlatParameters / flat_plan (mo-vae_b200/optim.py) and of the Jacobian buffer
bookkeeping in autojac.py.  The CUDA-only guard is lifted with a monkeypatch so that the pure tensor plumbing (offsets,
views, runs, adoption of foreign gradients) runs on CPU tensors; no kernel is called."""
import pytest
import torch
from torch import nn


@pytest.fixture()
def mv(monkeypatch):
    import movae_b200
    from movae_b200 import _lib

    monkeypatch.setattr(_lib, "require_cuda", lambda t, name: None)
    return movae_b200


def _net():
    torch.manual_seed(0)
    return nn.Sequential(nn.Conv2d(3, 5, 3), nn.Linear(7, 3), nn.Linear(3, 2, bias=False))     # numels 135, 5, 21, 3, 6


def test_layout_offsets_views_and_plan(mv):
    net = _net()
    before = [p.detach().clone() for p in net.parameters()]
    flat = mv.FlatParameters(net.parameters())
    assert flat.offsets == [0, 136, 144, 168, 172] and flat.total == 180          # every tensor starts on a multiple of 4
    for p, b, o in zip(net.parameters(), before, flat.offsets):
        assert torch.equal(p.detach(), b)
        assert p.data_ptr() == flat.flat_param.data_ptr() + 4 * o
    ps = list(net.parameters())
    ordered, cols, lo, hi = flat.plan([ps[2], ps[1]])                              # any order in, layout order out
    assert ordered == [ps[1], ps[2]] and cols == [0, 8] and (lo, hi) == (136, 168)
    assert flat.plan([ps[0], ps[2]]) is None                                       # not a consecutive run
    from movae_b200.optim import flat_plan

    assert flat_plan([ps[0], nn.Parameter(torch.zeros(2))]) is None                # a parameter outside the layout
    owner, ordered, cols, lo, hi = flat_plan(ps)
    assert owner is flat and (lo, hi) == (0, 180) and cols == flat.offsets
    with pytest.raises(RuntimeError):
        mv.FlatParameters(ps)                                                      # one layout per parameter


def test_gradient_adoption_runs_and_zero_grad(mv):
    net = _net()
    flat = mv.FlatParameters(net.parameters())
    ps = list(net.parameters())
    assert flat.gather_grads() == [] and all(flat.grad_state(p) == "none" for p in ps)
    ps[0].grad = torch.ones_like(ps[0])                                            # a foreign gradient (plain autograd)
    ps[1].grad = torch.full_like(ps[1], 2.0)
    ps[3].grad = torch.full_like(ps[3], 3.0)
    assert flat.grad_state(ps[0]) == "other"
    runs = flat.gather_grads()
    assert runs == [(0, 144), (168, 172)]                                          # params 0-1 contiguous, param 3 alone
    assert flat.runs([3, 0, 1]) == runs and flat.runs([]) == []
    assert flat.grad_state(ps[0]) == "view" and flat.grad_state(ps[2]) == "none"
    assert float(flat.flat_grad[:135].sum()) == 135.0 and float(flat.flat_grad[135]) == 0.0     # padding stays zero
    assert torch.equal(flat.flat_grad[136:141], torch.full((5,), 2.0)) and torch.equal(flat.flat_grad[168:171], torch.full((3,), 3.0))
    flat.adopt([ps[2]], [torch.full_like(ps[2], 4.0)])
    assert flat.grad_state(ps[2]) == "view" and float(ps[2].grad.sum()) == 84.0
    assert flat.gather_grads() == [(0, 172)]
    flat.zero_grad()
    assert all(p.grad is None for p in ps)
    flat.zero_grad(set_to_none=False)
    assert all(flat.grad_state(p) == "view" for p in ps) and float(flat.flat_grad.abs().sum()) == 0.0


def test_jacobian_buffer_is_cached_per_layout_and_padded(mv):
    from movae_b200 import autojac

    autojac._J_CACHE.clear()
    a = autojac._jacobian_buffer(3, 10, torch.device("cpu"))
    assert a.shape == (3, 10) and a.stride(0) == 12                                 # rows padded to 16 bytes
    assert autojac._jacobian_buffer(3, 10, torch.device("cpu")).data_ptr() == a.data_ptr()
    b = autojac._jacobian_buffer(3, 10, torch.device("cpu"), ("flat", 1, 0, 12), min_ld=24)     # data-parallel padding
    assert b.stride(0) == 24 and b.data_ptr() != a.data_ptr() and float(b.abs().sum()) == 0.0
    offs = autojac._dense_offsets([torch.zeros(3), torch.zeros(2, 2), torch.zeros(1)])
    assert offs == [0, 3, 7]
    J = autojac._jacobian_buffer(2, 8, torch.device("cpu"))
    params = [torch.zeros(3), torch.zeros(2, 2), torch.zeros(1)]
    autojac._fill_row(J, 1, params, [torch.ones(3), None, torch.full((1,), 5.0)], offs)
    assert J[1].tolist() == [1, 1, 1, 0, 0, 0, 0, 5] and float(J[0].abs().sum()) == 0.0
