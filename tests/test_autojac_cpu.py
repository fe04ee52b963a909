"""CPU tests of the Jacobian-descent engine (mo-vae_b200/autojac.py): `backward` and `mtl_backward` run through the
segmented and the flat-Jacobian paths with a stub aggregator of fixed weights written in plain torch, and their `.grad`
results are compared with gradients from torch.autograd.grad.  They pin where the aggregated gradient goes (torchjd's
Accumulate rule, on plain parameters and on every `.grad` state of a FlatParameters layout), that an objective which
never reaches the features costs no backward pass, and the order in which rows reach a data-parallel plan.  The
CUDA-only guard is lifted with a monkeypatch; no kernel is called."""
import pytest
import torch
from torch import nn

W = torch.tensor([0.5, -1.25, 2.0])      # the stub's weights: g = sum_i W[i] * row_i
ZERO_ROW = 1                             # the objective that never reaches the features
PATHS = pytest.mark.parametrize("segments", [True, False], ids=["segmented", "flat_jacobian"])
APIS = pytest.mark.parametrize("api", ["mtl_backward", "backward"])


@pytest.fixture()
def mv(monkeypatch):
    import movae_b200
    from movae_b200 import _lib

    monkeypatch.setattr(_lib, "require_cuda", lambda t, name: None)
    return movae_b200


@pytest.fixture()
def log(monkeypatch):
    """Events in call order; every torch.autograd.grad call adds ("grad",)."""
    events = []
    real = torch.autograd.grad

    def counted(*args, **kwargs):
        events.append(("grad",))
        return real(*args, **kwargs)

    monkeypatch.setattr(torch.autograd, "grad", counted)
    return events


class _Stub:
    """Aggregator with fixed weights; records which path called it and what it was given."""

    def __init__(self, segments: bool):
        self.segments = segments
        self.calls, self.rows, self.J = [], None, None

    def supports_segments(self):
        return self.segments

    def aggregate_segments_into(self, rows, numels, out_offsets, out, accumulate):
        self.calls.append("segments")
        self.rows = rows
        for s, (n, o) in enumerate(zip(numels, out_offsets)):
            g = W @ torch.stack([r[s].reshape(-1)[:n] for r in rows])
            out[o:o + n].add_(g) if accumulate else out[o:o + n].copy_(g)
        return W.clone()

    def aggregate_into(self, J, out, accumulate):
        self.calls.append("matrix")
        self.J = J.clone()
        out.add_(W @ J) if accumulate else out.copy_(W @ J)
        return W.clone()


class _RecordingDataParallel:
    """Stands in for parallel.DataParallel at world size 1 (averaging is the identity) and records its row protocol."""

    def __init__(self, log):
        self.log, self.rows, self.averaged = log, {}, []

    def padded_columns(self, P):
        return (P + 7) // 8 * 8 + 8

    def begin_rows(self, k, P, dtype, device):
        self.log.append(("begin",))
        self.k = k

    def row_ready(self, i, row_padded):
        self.log.append(("ready", i))
        self.rows[i] = row_padded.clone()

    def row_zero(self, i):
        self.log.append(("zero", i))
        self.rows[i] = None

    def aggregate_rows_into(self, P, out, accumulate):
        J = torch.stack([torch.zeros(P) if self.rows[i] is None else self.rows[i][:P] for i in range(self.k)])
        out.add_(W @ J) if accumulate else out.copy_(W @ J)
        return W.clone()

    def average_(self, tensors):
        self.averaged.append([(t.data_ptr(), t.numel()) for t in tensors])


class _Net(nn.Module):
    def __init__(self):
        super().__init__()
        torch.manual_seed(0)
        self.enc = nn.Sequential(nn.Linear(4, 6), nn.Tanh(), nn.Linear(6, 3))      # numels 24, 6, 18, 3: not all aligned
        self.h1 = nn.Linear(3, 2)
        self.h2 = nn.Linear(3, 1)
        self.code = nn.Parameter(torch.randn(3))
        self.x = torch.randn(5, 4)

    def forward(self):
        f = self.enc(self.x)
        l1 = self.h1(f).pow(2).mean()
        l2 = (self.code - f.detach().mean(0)).pow(2).mean()       # like an embedding loss: never reaches the features
        l3 = (self.h2(f) - 1).abs().mean() + 0.1 * self.code.sum()
        return f, [l1, l2, l3]


def _expected(net, api):
    """{parameter: the gradient one call of `api` gives it}, from torch.autograd.grad directly."""
    f, losses = net()
    shared = list(net.enc.parameters()) if api == "mtl_backward" else list(net.parameters())
    rows = []
    for l in losses:
        gs = torch.autograd.grad(l, shared, retain_graph=True, allow_unused=True)
        rows.append([torch.zeros_like(p) if g is None else g for p, g in zip(shared, gs)])
    out = {p: sum(w * r[j] for w, r in zip(W.tolist(), rows)) for j, p in enumerate(shared)}
    if api == "mtl_backward":                        # task-specific parameters: the plain sum of their losses' gradients
        heads = [p for p in net.parameters() if p not in out]
        out.update(zip(heads, torch.autograd.grad(sum(losses), heads)))
    return out


def _run(mv, api, net, agg):
    f, losses = net()
    if api == "mtl_backward":
        mv.mtl_backward(losses=losses, features=[f], aggregator=agg)
    else:
        mv.backward(losses, aggregator=agg, inputs=list(net.parameters()))


@PATHS
@APIS
def test_plain_parameters_are_assigned_then_added_to(mv, api, segments, log):
    net = _Net()
    exp = _expected(net, api)
    agg = _Stub(segments)
    _run(mv, api, net, agg)
    assert agg.calls == ["segments" if segments else "matrix"]
    for p, g in exp.items():
        torch.testing.assert_close(p.grad, g)
    before = {p: (p.grad, p.grad.clone()) for p in exp}
    _run(mv, api, net, agg)
    for p, g in exp.items():
        assert p.grad is before[p][0]                                    # added in place
        torch.testing.assert_close(p.grad, before[p][1] + g)


@pytest.mark.parametrize("state", ["none", "view", "mixed"])
@PATHS
@APIS
def test_flat_parameters_every_grad_state(mv, api, segments, state, log):
    net = _Net()
    exp = _expected(net, api)
    flat = mv.FlatParameters(net.parameters())
    ps = list(net.parameters())
    torch.manual_seed(1)
    if state != "none":
        flat.zero_grad(set_to_none=False)                                # every .grad a view of the flat gradient buffer
        for p in ps:
            p.grad.copy_(torch.randn_like(p))
    if state == "mixed":                                                 # none / view / a tensor living elsewhere, in turn
        for i, p in enumerate(ps):
            p.grad = None if i % 3 == 0 else p.grad if i % 3 == 1 else torch.randn_like(p)
    before = {p: (p.grad, None if p.grad is None else p.grad.clone(), flat.grad_state(p)) for p in ps}
    padding = torch.ones(flat.total, dtype=torch.bool)
    for o, p in zip(flat.offsets, ps):
        padding[o:o + p.numel()] = False
    agg = _Stub(segments)
    _run(mv, api, net, agg)
    assert agg.calls == ["segments" if segments else "matrix"]
    for p, g in exp.items():
        obj, old, st = before[p]
        if old is None:
            torch.testing.assert_close(p.grad, g)
        else:
            assert p.grad is obj
            torch.testing.assert_close(p.grad, old + g)
        if st == "view" or state == "none":
            assert flat.grad_state(p) == "view"
    assert float(flat.flat_grad[padding].abs().sum()) == 0.0


@PATHS
def test_objective_that_never_reaches_the_features_costs_no_backward_pass(mv, segments, log):
    from movae_b200 import autojac

    net = _Net()
    exp = _expected(net, "mtl_backward")
    agg = _Stub(segments)
    _run(mv, "mtl_backward", net, agg)
    for buf in autojac._J_CACHE.values():                                # a stale row left by an earlier step
        buf[ZERO_ROW].fill_(float("nan"))
    for p in net.parameters():
        p.grad = None
    log.clear()
    _run(mv, "mtl_backward", net, agg)
    assert len(log) == 3 + 2                         # one pass per loss to the features, one per row that reaches them
    if segments:
        zero = autojac._ZEROS[torch.device("cpu")]
        assert len(agg.rows) == 3 and all(t.data_ptr() == zero.data_ptr() for t in agg.rows[ZERO_ROW])
    else:
        assert agg.J.shape[0] == 3 and float(agg.J[ZERO_ROW].abs().sum()) == 0.0
    for p, g in exp.items():
        torch.testing.assert_close(p.grad, g)


@pytest.mark.parametrize("flat", [False, True], ids=["plain", "flat_parameters"])
@APIS
def test_data_parallel_gets_each_row_between_backward_passes(mv, api, flat, log):
    net = _Net()
    exp = _expected(net, api)
    fp = mv.FlatParameters(net.parameters()) if flat else None
    agg = _Stub(True)
    agg.data_parallel = dp = _RecordingDataParallel(log)
    log.clear()
    _run(mv, api, net, agg)
    assert agg.calls == []                                               # the plan aggregates the rows it was handed
    for p, g in exp.items():
        torch.testing.assert_close(p.grad, g)
    mtl = api == "mtl_backward"
    b = log.index(("begin",))
    assert log[:b] == [("grad",)] * (3 if mtl else 0)                    # mtl_backward: the feature / task gradients
    live = [0, 2] if mtl else [0, 1, 2]
    assert [e for e in log[b + 1:] if e[0] != "zero"] == [e for i in live for e in (("grad",), ("ready", i))]
    assert [e[1] for e in log if e[0] == "zero"] == ([ZERO_ROW] if mtl else [])
    # layout order: code (3 -> 4 columns), enc (24, 8, 20, 4), h1 (8, 4), h2 (4, 4); 80 columns in all
    shared = list(net.enc.parameters()) if mtl else list(net.parameters())
    P = (56 if mtl else 80) if flat else sum(p.numel() for p in shared)
    for i in live:
        assert dp.rows[i].numel() == dp.padded_columns(P)
        assert float(dp.rows[i][P:].abs().sum()) == 0.0                  # the padding columns carry zeros
    if not mtl:
        assert dp.averaged == []
    elif flat:                                                           # the fresh task gradients: [lo, hi) runs of the buffer
        base = fp.flat_grad.data_ptr()
        assert [[((a - base) // 4, n) for a, n in runs] for runs in dp.averaged] == [[(0, 4), (60, 20)]]
    else:                                                                # one average per task-specific parameter
        assert sorted(n for a in dp.averaged for _, n in a) == sorted(p.numel() for p in exp if all(p is not s for s in shared))
