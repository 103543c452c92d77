"""Every optimizer variant and NCCL-style baseline is equivalent to single-process SGD."""
import pytest
import torch
import torch.nn as nn

from _mp import run_ranks
from test_dear_equivalence import data, make_model, reference_run

CASE = dict(momentum=0.9, weight_decay=1e-3)


def worker(rank, world, kind, steps, per_rank):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.parallel import variants
    from dear_pytorch_b200.parallel.baselines import WFBPDistributedOptimizer, wrap_ddp
    from dear_pytorch_b200.parallel.baselines import ByteSchedulerOptimizer, HorovodOptimizer
    from dear_pytorch_b200.utils.profiling import benchmark
    model = make_model()
    model.eval()
    opt = torch.optim.SGD(model.parameters(), lr=0.05, **CASE)
    fwd = model
    if kind == "naive":
        opt = variants.NaiveDistributedOptimizer(opt, model, verbose=False)
    elif kind == "wt":
        opt = variants.WaitTimeDistributedOptimizer(opt, model, cycle_time_ms=0.05, warmup_steps=2, verbose=False)
    elif kind == "rb":
        opt = variants.ReduceBroadcastDistributedOptimizer(opt, model, threshold=0.002, verbose=False)
    elif kind == "wfbp":
        opt = WFBPDistributedOptimizer(opt, model=model, threshold=0, verbose=False)
    elif kind == "wfbp-threshold":
        opt = WFBPDistributedOptimizer(opt, model=model, threshold=600, verbose=False)
    elif kind in ("mgwfbp", "asc"):
        x, y = data(0, 4)
        seq, times, sizes = benchmark(model, (x, y), nn.functional.cross_entropy, warmup=1, iters=2)
        seq, times = dear.runtime.broadcast_object((seq, times), src=0)
        opt = WFBPDistributedOptimizer(opt, model=model, seq_layernames=seq, layerwise_times=times, mgwfbp=(kind == "mgwfbp"),
                                       asc=(kind == "asc"), alpha=1e-4, beta=1e-9, verbose=False)
    elif kind == "horovod":
        opt = HorovodOptimizer(opt, model, cycle_time_ms=0.2, fusion_threshold_mb=0.002, negotiation_steps=2, verbose=False)
    elif kind == "bytescheduler":
        opt = ByteSchedulerOptimizer(opt, model, partition=100, credit=250, verbose=False)
    elif kind in ("ddp", "ddp-zero"):
        fwd, opt = wrap_ddp(model, torch.optim.SGD, dict(lr=0.05, **CASE), zero=(kind == "ddp-zero"))
    if kind not in ("ddp", "ddp-zero"):
        dear.broadcast_parameters(model.state_dict(), 0)
    for t in range(steps):
        x, y = data(t, world * per_rank)
        x, y = x[rank * per_rank:(rank + 1) * per_rank], y[rank * per_rank:(rank + 1) * per_rank]
        opt.zero_grad()
        nn.functional.cross_entropy(fwd(x), y).backward()
        opt.step()
    if hasattr(opt, "synchronize") and kind in ("naive", "wt", "rb", "bytescheduler"):
        opt.synchronize()
    info = None
    if kind == "wt":
        info = (opt.wait_time.done, len(opt.engine.plan.buckets))
    elif kind == "horovod":
        info = (opt.groups, len(list(model.parameters())))
    elif kind == "bytescheduler":
        info = (list(opt.launch_log), opt.partition, opt.credit)
    return [p.detach().clone() for p in model.parameters()], info


@pytest.mark.parametrize("kind", ["naive", "wt", "rb", "wfbp", "wfbp-threshold", "mgwfbp", "asc", "horovod",
                                  "bytescheduler", "ddp", "ddp-zero"])
def test_variant_matches_sgd(kind):
    steps, per_rank, world = 5, 3, 2
    ref = reference_run(CASE, steps, world, per_rank)
    outs = run_ranks(worker, world=world, backend="gloo", args=(kind, steps, per_rank))
    for params, info in outs:
        for a, b in zip(params, ref):
            torch.testing.assert_close(a, b, rtol=3e-5, atol=3e-6)
        if kind == "wt":
            assert info[0] and info[1] >= 1
        if kind == "horovod":
            groups, ntensors = info
            assert groups is not None and sum(len(g) for g in groups) == ntensors      # response cache was built
            assert groups == outs[0][1][0]                                             # identical on every rank
        if kind == "bytescheduler":
            log, partition, credit = info
            assert log == outs[0][1][0]                                                # same collective order on every rank
            assert max(n for _, _, n in log) <= partition and any(i > 0 for _, i, _ in log)   # tensors were partitioned


def _wfbp_timers_worker(rank, world):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.parallel.baselines import WFBPDistributedOptimizer
    model = make_model()
    opt = WFBPDistributedOptimizer(torch.optim.SGD(model.parameters(), lr=0.05), model=model, compression="topk",
                                   is_sparse=True, density=0.25, threshold=600, profiling=True, verbose=False)
    dear.broadcast_parameters(model.state_dict(), 0)
    for t in range(2):
        x, y = data(t, 8)
        opt.zero_grad()
        nn.functional.cross_entropy(model(x[rank * 4:(rank + 1) * 4]), y[rank * 4:(rank + 1) * 4]).backward()
        opt.step()
    return opt.profiling_summary()


def test_wfbp_in_optimizer_timers():
    out = run_ranks(_wfbp_timers_worker, world=2, backend="gloo")[0]
    assert out["compression"] and set(out["compression"]) == set(out["allreduce"]) == set(out["update"])
    assert all(v > 0 for v in out["allreduce"].values())


def test_horovod_cycle_grouping():
    from dear_pytorch_b200.parallel.baselines import cycle_groups
    t = [0.0, 1.0, 4.9, 5.1, 6.0, 20.0]                    # ms since the first gradient
    nb = [10, 10, 10, 10, 10, 10]
    assert cycle_groups(t, nb, 5.0, 1 << 20) == [[0, 1, 2], [3, 4], [5]]           # cut at cycle boundaries
    assert cycle_groups(t, nb, 5.0, 25) == [[0, 1], [2], [3, 4], [5]]              # ... and at the fusion threshold
    assert cycle_groups(t, nb, 0.0, 1 << 20) == [[i] for i in range(6)]            # HOROVOD_CYCLE_TIME=0: no fusion
    assert cycle_groups(t, [100] * 6, 5.0, 50) == [[i] for i in range(6)]          # oversized tensors travel alone


def test_bytescheduler_priority_and_credit():
    """Single process, fake collectives: chunks leave in forward-priority order under the credit."""
    import heapq
    from dear_pytorch_b200.parallel.baselines import partition_sizes
    from dear_pytorch_b200.parallel.baselines.bytescheduler import _Chunk
    assert partition_sizes(10, 4) == [4, 4, 2] and partition_sizes(3, 4) == [3] and partition_sizes(8, 0) == [8]
    heap = []
    for prio, n in [(5, 3), (2, 2), (7, 1), (0, 2)]:           # arrival order = backward order (last layers first)
        for i in range(n):
            heapq.heappush(heap, _Chunk(prio, i, torch.zeros(1), None))
    order = [(c.prio, c.idx) for c in (heapq.heappop(heap) for _ in range(len(heap)))]
    assert order == [(0, 0), (0, 1), (2, 0), (2, 1), (5, 0), (5, 1), (5, 2), (7, 0)]


def _sparse_consistency_worker(rank, world, compressor, mc):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.parallel.baselines import WFBPDistributedOptimizer
    model = make_model()
    opt = torch.optim.SGD(model.parameters(), lr=0.05, momentum=0.9 if mc else 0.0)
    opt = WFBPDistributedOptimizer(opt, model=model, compression=compressor, is_sparse=True, density=0.25,
                                   threshold=10 ** 9, momentum_correction=mc, verbose=False)
    dear.broadcast_parameters(model.state_dict(), 0)
    losses = []
    for t in range(8):
        x, y = data(0, 8)
        opt.zero_grad()
        loss = nn.functional.cross_entropy(model(x[rank * 4:(rank + 1) * 4]), y[rank * 4:(rank + 1) * 4])
        loss.backward()
        opt.step()
        losses.append(float(loss))
    return losses, [p.detach().clone() for p in model.parameters()]


@pytest.mark.parametrize("compressor,mc", [("gtopk", False), ("gtopkef", False), ("topk", True), ("gaussian", False)])
def test_sparse_paths_stay_rank_consistent(compressor, mc):
    outs = run_ranks(_sparse_consistency_worker, world=2, backend="gloo", args=(compressor, mc))
    assert all(torch.equal(a, b) for a, b in zip(outs[0][1], outs[1][1]))
    assert outs[0][0][-1] < outs[0][0][0]            # the sparsified run still trains


def _sparse_topk_allgather_worker(rank, world):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.parallel.baselines import WFBPDistributedOptimizer
    model = make_model()
    opt = torch.optim.SGD(model.parameters(), lr=0.05)
    opt = WFBPDistributedOptimizer(opt, model=model, compression="topk", is_sparse=True, density=0.25, threshold=0,
                                   verbose=False)
    dear.broadcast_parameters(model.state_dict(), 0)
    losses = []
    for t in range(6):
        x, y = data(0, 8)
        opt.zero_grad()
        loss = nn.functional.cross_entropy(model(x[rank * 4:(rank + 1) * 4]), y[rank * 4:(rank + 1) * 4])
        loss.backward()
        opt.step()
        losses.append(float(loss))
    return losses, [p.detach().clone() for p in model.parameters()]


def test_sparse_topk_allgather_path_runs():
    outs = run_ranks(_sparse_topk_allgather_worker, world=2, backend="gloo")
    assert all(torch.equal(a, b) for a, b in zip(outs[0][1], outs[1][1]))
    assert outs[0][0][-1] < outs[0][0][0] + 0.5


def _adasum_worker(rank, world, mode):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.parallel.baselines import HorovodOptimizer
    torch.manual_seed(0)
    model = nn.Linear(world, 1, bias=False)
    with torch.no_grad():
        model.weight.zero_()
    opt = HorovodOptimizer(torch.optim.SGD(model.parameters(), lr=1.0), model, op="adasum", negotiation_steps=1, verbose=False)
    moved = []
    for step in range(3):                                   # step 0: cold cache (per tensor), later: fused buffer
        opt.zero_grad()
        if mode == "orthogonal":
            x = torch.zeros(1, world); x[0, rank] = 1.0      # d loss / d w = e_rank on every rank
        else:
            x = torch.ones(1, world) * 0.5                   # the same gradient on every rank
        before = model.weight.detach().clone()
        model(x).sum().backward()
        opt.step()
        moved.append((before - model.weight.detach()).flatten())
    return moved


@pytest.mark.parametrize("world", [2, 4])
def test_horovod_adasum_adds_orthogonal_and_averages_parallel_gradients(world):
    for mode, expect in (("orthogonal", torch.ones(world)), ("parallel", torch.full((world,), 0.5))):
        outs = run_ranks(_adasum_worker, world=world, backend="gloo", args=(mode,))
        for moved in outs:
            for m in moved:
                torch.testing.assert_close(m, expect)
        assert all(torch.equal(a, b) for a, b in zip(outs[0], outs[-1]))       # bit-identical on every rank


def _adasum_three_ranks_worker(rank, world):
    from dear_pytorch_b200.parallel.baselines import HorovodOptimizer
    m = nn.Linear(2, 2)
    try:
        HorovodOptimizer(torch.optim.SGD(m.parameters(), lr=1.0), m, op="adasum", verbose=False)
    except ValueError as e:
        return str(e)
    return None


def test_adasum_needs_a_power_of_two():
    assert all("power-of-two" in (o or "") for o in run_ranks(_adasum_three_ranks_worker, world=3, backend="gloo"))


def _fp16_worker(rank, world):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.parallel.baselines import HorovodOptimizer
    model = make_model()
    model.eval()
    opt = HorovodOptimizer(torch.optim.SGD(model.parameters(), lr=0.05, **CASE), model, fp16_allreduce=True,
                           cycle_time_ms=0.2, fusion_threshold_mb=0.002, negotiation_steps=2, verbose=False)
    dear.broadcast_parameters(model.state_dict(), 0)
    for t in range(4):
        x, y = data(t, world * 3)
        opt.zero_grad()
        nn.functional.cross_entropy(model(x[rank * 3:(rank + 1) * 3]), y[rank * 3:(rank + 1) * 3]).backward()
        opt.step()
    return [p.detach().clone() for p in model.parameters()]


def test_horovod_fp16_allreduce_tracks_fp32_within_half_precision():
    ref = reference_run(CASE, 4, 2, 3)
    outs = run_ranks(_fp16_worker, world=2, backend="gloo")
    exact = True
    for a, b in zip(outs[0], ref):
        torch.testing.assert_close(a, b, rtol=5e-3, atol=5e-4)
        exact = exact and torch.equal(a, b)
    assert not exact                                             # the wire really was fp16
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)


def _rb_unused_worker(rank, world, steps, per_rank):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.parallel import variants
    from test_stress_order import Tangled, batch
    m = Tangled(depth=3)
    opt = variants.ReduceBroadcastDistributedOptimizer(torch.optim.SGD(m.parameters(), lr=0.05, momentum=0.9, weight_decay=1e-3),
                                                       m, threshold=0.002, verbose=False)
    dear.broadcast_parameters(m.state_dict(), 0)
    for t in range(steps):
        x, y = batch(t, world * per_rank)
        opt.zero_grad()
        nn.functional.cross_entropy(m(x[rank * per_rank:(rank + 1) * per_rank]), y[rank * per_rank:(rank + 1) * per_rank]).backward()
        opt.step()
    opt.synchronize()
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def test_reduce_broadcast_variant_leaves_unused_parameters_alone():
    """``Tangled.unused`` never runs: with weight decay + momentum torch.optim does not touch it (its gradient is None);
    the variant's bucket-view gradients are all zeros there and must not be treated as a gradient."""
    from test_stress_order import Tangled, batch
    steps, world, per = 4, 2, 2
    ref = Tangled(depth=3)
    opt = torch.optim.SGD(ref.parameters(), lr=0.05, momentum=0.9, weight_decay=1e-3)
    w0 = ref.unused.weight.detach().clone()
    for t in range(steps):
        x, y = batch(t, world * per)
        opt.zero_grad()
        nn.functional.cross_entropy(ref(x), y).backward()
        opt.step()
    assert torch.equal(ref.unused.weight, w0)
    for sd in run_ranks(_rb_unused_worker, world=world, backend="gloo", args=(steps, per)):
        for k, v in ref.state_dict().items():
            torch.testing.assert_close(sd[k], v, rtol=3e-5, atol=3e-6)


def _bsc_sched_worker(rank, world, steps, per_rank):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.parallel.baselines import ByteSchedulerOptimizer
    model = make_model()
    model.eval()
    opt = ByteSchedulerOptimizer(torch.optim.SGD(model.parameters(), lr=0.05, **CASE), model, partition=100, credit=250, verbose=False)
    sched = torch.optim.lr_scheduler.StepLR(opt, 1, 0.5)
    dear.broadcast_parameters(model.state_dict(), 0)
    for t in range(steps):
        x, y = data(t, world * per_rank)
        opt.zero_grad()
        nn.functional.cross_entropy(model(x[rank * per_rank:(rank + 1) * per_rank]), y[rank * per_rank:(rank + 1) * per_rank]).backward()
        opt.step()
        sched.step()                 # changes the lr BEFORE the deferred per-layer updates of this step are applied
    opt.synchronize()
    return [p.detach().clone() for p in model.parameters()]


def test_bytescheduler_deferred_updates_use_the_lr_of_their_own_step():
    steps, per_rank, world = 4, 3, 2
    model = make_model()
    model.eval()
    opt = torch.optim.SGD(model.parameters(), lr=0.05, **CASE)
    sched = torch.optim.lr_scheduler.StepLR(opt, 1, 0.5)
    for t in range(steps):
        x, y = data(t, world * per_rank)
        opt.zero_grad()
        nn.functional.cross_entropy(model(x), y).backward()
        opt.step()
        sched.step()
    for params in run_ranks(_bsc_sched_worker, world=world, backend="gloo", args=(steps, per_rank)):
        for a, b in zip(params, model.parameters()):
            torch.testing.assert_close(a, b.detach(), rtol=3e-5, atol=3e-6)


def _lossless_sparse_worker(rank, world, comp, mc):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.parallel.baselines import WFBPDistributedOptimizer
    m = make_model(); m.eval()
    opt = WFBPDistributedOptimizer(torch.optim.SGD(m.parameters(), lr=0.05, momentum=0.9), model=m, compression=comp, is_sparse=True,
                                   density=1.0, threshold=600, momentum_correction=mc, verbose=False)
    dear.broadcast_parameters(m.state_dict(), 0)
    for t in range(4):
        x, y = data(t, 4)
        opt.zero_grad()
        nn.functional.cross_entropy(m(x[rank * 2:(rank + 1) * 2]), y[rank * 2:(rank + 1) * 2]).backward()
        opt.step()
    return [p.detach().clone() for p in m.parameters()]


@pytest.mark.parametrize("mc", [False, True])
@pytest.mark.parametrize("comp", ["topk", "eftopk", "gtopk", "gtopkef"])
def test_sparse_path_at_density_one_is_the_dense_optimizer(comp, mc):
    """Invariant: selecting every element loses nothing, so the sparse all-gather / gTop-k path — with or without momentum
    correction, whose factor masking only applies below density 1 (wfbp/dopt.py:948) — must reproduce momentum SGD."""
    ref = reference_run(dict(momentum=0.9), 4, 2, 2)
    for params in run_ranks(_lossless_sparse_worker, world=2, backend="gloo", args=(comp, mc)):
        for a, b in zip(params, ref):
            torch.testing.assert_close(a, b, rtol=3e-5, atol=3e-6)
