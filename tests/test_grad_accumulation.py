"""backward_passes_per_step=k: gradients accumulate locally over k backward passes, the reduce-scatter runs during
the k-th, one step() per k passes — equal to one pass over the concatenated micro-batches."""
import pytest
import torch
import torch.nn as nn

from _mp import run_ranks
from test_dear_equivalence import data, make_model, reference_run


class SometimesUnused(nn.Module):
    """`extra` takes part only in even micro-batches: it sees fewer passes than backward_passes_per_step."""

    def __init__(self):
        super().__init__()
        torch.manual_seed(3)
        self.a = nn.Linear(6, 6)
        self.extra = nn.Linear(6, 6)
        self.b = nn.Linear(6, 3)

    def forward(self, x, use_extra):
        h = torch.tanh(self.a(x))
        if use_extra:
            h = h + torch.tanh(self.extra(h))
        return self.b(h)


def worker(rank, world, case, steps, per_rank, k):
    import dear_pytorch_b200 as dear
    model = make_model(); model.eval()
    opt = torch.optim.SGD(model.parameters(), lr=0.05, **case)
    opt = dear.DistributedOptimizer(opt, model, threshold=0.001, verbose=False, backward_passes_per_step=k)
    dear.broadcast_parameters(model.state_dict(), 0)
    micro = per_rank // k
    for t in range(steps):
        x, y = data(t, world * per_rank)
        x, y = x[rank * per_rank:(rank + 1) * per_rank], y[rank * per_rank:(rank + 1) * per_rank]
        opt.zero_grad()
        for j in range(k):
            xs, ys = x[j * micro:(j + 1) * micro], y[j * micro:(j + 1) * micro]
            (nn.functional.cross_entropy(model(xs), ys) / k).backward()
        opt.step()
    opt.synchronize()
    return [p.detach().clone() for p in model.parameters()]


@pytest.mark.parametrize("backend", ["gloo", "emu"])
@pytest.mark.parametrize("k", [2, 4])
def test_accumulation_equals_one_large_batch(backend, k):
    case = dict(momentum=0.9, weight_decay=1e-3)
    steps, world, per_rank = 3, 2, 4
    ref = reference_run(case, steps, world, per_rank)
    for params in run_ranks(worker, world=world, backend=backend, args=(case, steps, per_rank, k)):
        for a, b in zip(params, ref):
            torch.testing.assert_close(a, b, rtol=5e-5, atol=5e-6)


def gpu_worker(rank, world, case, steps, per_rank, k):
    import dear_pytorch_b200 as dear
    dev = dear.device()
    model = make_model().to(dev); model.eval()
    opt = torch.optim.SGD(model.parameters(), lr=0.05, **case)
    opt = dear.DistributedOptimizer(opt, model, threshold=0.001, verbose=False, backward_passes_per_step=k)
    dear.broadcast_parameters(model.state_dict(), 0)
    micro = per_rank // k
    for t in range(steps):
        x, y = data(t, world * per_rank)
        x, y = x[rank * per_rank:(rank + 1) * per_rank].to(dev), y[rank * per_rank:(rank + 1) * per_rank].to(dev)
        for j in range(k):
            (nn.functional.cross_entropy(model(x[j * micro:(j + 1) * micro]), y[j * micro:(j + 1) * micro]) / k).backward()
        opt.step()
    opt.synchronize()
    dear.communicator().check_status()
    return [p.detach().cpu() for p in model.parameters()]


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
def test_accumulation_on_gpu(world):
    case = dict(momentum=0.9, weight_decay=1e-3)
    ref = reference_run(case, 3, world, 4)
    for params in run_ranks(gpu_worker, world=world, backend="b200", args=(case, 3, 4, 2),
                            extra_env={"DEAR_SPIN_TIMEOUT_S": "15"}, timeout=300):
        for a, b in zip(params, ref):
            torch.testing.assert_close(a, b, rtol=2e-4, atol=5e-6)


def unused_worker(rank, world, k):
    import dear_pytorch_b200 as dear
    model = SometimesUnused()
    opt = dear.DistributedOptimizer(torch.optim.SGD(model.parameters(), lr=0.1), model, threshold=None, num_nearby_layers=-1,
                                    verbose=False, backward_passes_per_step=k)
    dear.broadcast_parameters(model.state_dict(), 0)
    g = torch.Generator().manual_seed(5)
    xs = [torch.randn(4 * world, 6, generator=g) for _ in range(2 * k)]
    for t in range(2):
        opt.zero_grad()
        for j in range(k):
            x = xs[t * k + j][rank * 4:(rank + 1) * 4]
            (model(x, use_extra=(j % 2 == 0)).square().mean() / k).backward()
        opt.step()
    opt.synchronize()
    return [p.detach().clone() for p in model.parameters()], xs


@pytest.mark.parametrize("backend", ["gloo", "emu"])
def test_parameter_used_in_only_some_passes(backend):
    k, world = 2, 2
    outs = run_ranks(unused_worker, world=world, backend=backend, args=(k,))
    xs = outs[0][1]
    ref = SometimesUnused()
    opt = torch.optim.SGD(ref.parameters(), lr=0.1)
    for t in range(2):
        opt.zero_grad()
        for j in range(k):
            # mean over the global micro-batch == mean over ranks of the per-rank means (equal shard sizes)
            (ref(xs[t * k + j], use_extra=(j % 2 == 0)).square().mean() / k).backward()
        opt.step()
    for params, _ in outs:
        for a, b in zip(params, ref.parameters()):
            torch.testing.assert_close(a, b.detach(), rtol=5e-5, atol=5e-6)


def _second_backward_worker(rank, world):
    import dear_pytorch_b200 as dear
    model = make_model(); model.eval()
    opt = dear.DistributedOptimizer(torch.optim.SGD(model.parameters(), lr=0.1), model, threshold=0.001, verbose=False)
    x, y = data(0, 4)
    nn.functional.cross_entropy(model(x), y).backward()
    try:
        nn.functional.cross_entropy(model(x), y).backward()
    except RuntimeError as e:
        return "backward_passes_per_step" in str(e)
    return False


def test_second_backward_without_accumulation_is_an_error():
    assert all(run_ranks(_second_backward_worker, world=1, backend="gloo"))


def _intermittent_worker(rank, world, steps, k, per):
    import dear_pytorch_b200 as dear
    from test_adam import _Branchy, _branchy_data
    m = _Branchy()
    opt = dear.DistributedOptimizer(torch.optim.SGD(m.parameters(), lr=0.05, momentum=0.9, weight_decay=1e-2), m,
                                    threshold=0.0005, backward_passes_per_step=k, verbose=False)
    dear.broadcast_parameters(m.state_dict(), 0)
    for t in range(steps):
        opt.zero_grad()
        for a in range(k):
            x, y = _branchy_data(t * k + a, world * per)
            (nn.functional.cross_entropy(m(x[rank * per:(rank + 1) * per], (t * k + a) % 5 == 1), y[rank * per:(rank + 1) * per]) / k).backward()
        opt.step()
    opt.synchronize()
    return [p.detach().clone() for p in m.parameters()]


@pytest.mark.parametrize("backend", ["gloo", "emu"])
def test_accumulation_with_a_branch_that_skips_whole_steps(backend):
    """k = 3 passes per step, the side branch runs in passes 1 and 6 only: step 0 and step 2 accumulate its gradient
    over fewer passes than k, step 1 has none at all — there torch.optim leaves the parameter (and its momentum) alone.
    In bucket-view mode ``p.grad`` stays allocated between steps, so "no gradient" has to come from the hook count."""
    from test_adam import _Branchy, _branchy_data
    steps, k, world, per = 3, 3, 2, 2
    ref = _Branchy()
    opt = torch.optim.SGD(ref.parameters(), lr=0.05, momentum=0.9, weight_decay=1e-2)
    for t in range(steps):
        opt.zero_grad()
        for a in range(k):
            x, y = _branchy_data(t * k + a, world * per)
            (nn.functional.cross_entropy(ref(x, (t * k + a) % 5 == 1), y) / k).backward()
        opt.step()
    for params in run_ranks(_intermittent_worker, world=world, backend=backend, args=(steps, k, per)):
        for a, b in zip(params, ref.parameters()):
            torch.testing.assert_close(a, b.detach(), rtol=3e-5, atol=3e-6)
