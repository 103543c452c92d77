"""``DistributedOptimizer(..., norm_clip=c)``: global-norm clipping of the averaged gradients on the sharded path ==
``torch.nn.utils.clip_grad_norm_`` before ``optimizer.step()`` (the reference's DeAR factory accepts the argument and
ignores it, dear/dear_dopt.py:381-398; its WFBP optimizer clips per tensor, wfbp/dopt.py:855-862)."""
import pytest
import torch
import torch.nn as nn

from _mp import run_ranks
from test_dear_equivalence import data, make_model


def _make(kind, params):
    if kind == "sgd":
        return torch.optim.SGD(params, lr=0.05, momentum=0.9, weight_decay=1e-3)
    return torch.optim.AdamW(params, lr=0.01)


def _reference(kind, clip, steps, n):
    m = make_model(); m.eval()
    opt = _make(kind, m.parameters())
    norms = []
    for t in range(steps):
        x, y = data(t, n)
        opt.zero_grad()
        nn.functional.cross_entropy(m(x), y).backward()
        norms.append(float(torch.nn.utils.clip_grad_norm_(m.parameters(), clip)))
        opt.step()
    return [p.detach().clone() for p in m.parameters()], norms


def clip_worker(rank, world, kind, clip, steps, n, to_device=False):
    import dear_pytorch_b200 as dear
    dev = dear.device()
    m = make_model().to(dev); m.eval()
    opt = dear.DistributedOptimizer(_make(kind, m.parameters()), m, threshold=0.001, norm_clip=clip, verbose=False)
    dear.broadcast_parameters(m.state_dict(), 0)
    per = n // world
    norms = []
    for t in range(steps):
        x, y = data(t, n)
        opt.zero_grad()
        nn.functional.cross_entropy(m(x[rank * per:(rank + 1) * per].to(dev)), y[rank * per:(rank + 1) * per].to(dev)).backward()
        opt.step()
        norms.append(float(opt.engine.last_grad_norm))
    opt.synchronize()
    return [p.detach().float().cpu().clone() for p in m.parameters()], norms


@pytest.mark.parametrize("backend,world", [("emu", 2), ("gloo", 3)])
@pytest.mark.parametrize("kind,clip", [("sgd", 0.5), ("adamw", 0.5), ("sgd", 100.0)])
def test_norm_clip_matches_clip_grad_norm(backend, world, kind, clip):
    steps, n = 5, 6
    ref, ref_norms = _reference(kind, clip, steps, n)
    assert (max(ref_norms) > clip) == (clip < 1.0)              # 0.5 really clips, 100 never does
    for params, norms in run_ranks(clip_worker, world=world, backend=backend, args=(kind, clip, steps, n)):
        torch.testing.assert_close(torch.tensor(norms), torch.tensor(ref_norms), rtol=1e-5, atol=1e-6)
        for a, b in zip(params, ref):
            torch.testing.assert_close(a, b, rtol=2e-5, atol=2e-6)


def _zero_clip_worker(rank, world):
    import dear_pytorch_b200 as dear
    m = nn.Linear(2, 2)
    try:
        dear.DistributedOptimizer(torch.optim.SGD(m.parameters(), lr=0.1), m, norm_clip=0.0, verbose=False)
    except ValueError as e:
        return str(e)


def test_norm_clip_rejects_nonsense():
    assert all("positive" in (o or "") for o in run_ranks(_zero_clip_worker, world=2, backend="emu"))
