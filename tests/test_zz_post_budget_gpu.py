"""GPU runs of everything that was written AFTER the round's GPU budget was spent (profiles/README.md R2.0).

These features were developed against the CPU backends only — same Python engine, same C++ runtime, kernels emulated on
the host — and have never executed on hardware by the time they were committed.  The file sorts last on purpose: whatever
happens here cannot hide the result of a test that ran on hardware before.  Ranks share one GPU through CUDA IPC when the
box has only one."""
import pytest
import torch
import torch.nn as nn

from _mp import run_ranks
from test_dear_equivalence import data, make_model

pytestmark = pytest.mark.gpu
ENV = {"DEAR_SPIN_TIMEOUT_S": "15"}


def _world():
    return 2 if torch.cuda.device_count() in (1, 2, 4, 8) else 1


# ---- global-norm clipping on the sharded path ---------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["sgd", "adamw"])
def test_norm_clip_on_the_fused_kernels(kind):
    from test_grad_clip import _reference, clip_worker
    steps, n, clip = 4, 8, 0.5
    ref, ref_norms = _reference(kind, clip, steps, n)
    for params, norms in run_ranks(clip_worker, world=_world(), backend="b200", args=(kind, clip, steps, n), extra_env=ENV, timeout=300):
        torch.testing.assert_close(torch.tensor(norms), torch.tensor(ref_norms), rtol=1e-4, atol=1e-5)
        for a, b in zip(params, ref):
            torch.testing.assert_close(a, b, rtol=2e-4, atol=2e-5)


# ---- per-parameter Adam step counts / late-starting momentum buffers -------------------------------------------------------
def _branchy_gpu_worker(rank, world, kind, steps, per):
    import dear_pytorch_b200 as dear
    from test_adam import _Branchy, _branchy_data
    dev = dear.device()
    m = _Branchy().to(dev)
    if kind == "adam":
        base = torch.optim.Adam(m.parameters(), lr=1e-2, weight_decay=1e-2)
    else:
        base = torch.optim.SGD(m.parameters(), lr=0.05, momentum=0.8, dampening=0.3, weight_decay=5e-3)
    opt = dear.DistributedOptimizer(base, m, threshold=0.0005, verbose=False)
    dear.broadcast_parameters(m.state_dict(), 0)
    for t in range(steps):
        x, y = _branchy_data(t, world * per)
        opt.zero_grad()
        nn.functional.cross_entropy(m(x[rank * per:(rank + 1) * per].to(dev), t % 3 == 2), y[rank * per:(rank + 1) * per].to(dev)).backward()
        opt.step()
    opt.synchronize()
    dear.communicator().check_status()
    return [p.detach().float().cpu() for p in m.parameters()]


@pytest.mark.parametrize("kind", ["adam", "sgd-dampening"])
def test_conditionally_executed_branch_matches_torch_optim(kind):
    from test_adam import _Branchy, _branchy_data
    steps, per, world = 7, 2, _world()
    ref = _Branchy()
    if kind == "adam":
        opt = torch.optim.Adam(ref.parameters(), lr=1e-2, weight_decay=1e-2)
    else:
        opt = torch.optim.SGD(ref.parameters(), lr=0.05, momentum=0.8, dampening=0.3, weight_decay=5e-3)
    for t in range(steps):
        x, y = _branchy_data(t, world * per)
        opt.zero_grad()
        nn.functional.cross_entropy(ref(x, t % 3 == 2), y).backward()
        opt.step()
    for params in run_ranks(_branchy_gpu_worker, world=world, backend="b200", args=(kind, steps, per), extra_env=ENV, timeout=300):
        for a, b in zip(params, ref.parameters()):
            torch.testing.assert_close(a, b.detach(), rtol=1e-3, atol=2e-5)


# ---- direct wgrad under autocast ------------------------------------------------------------------------------------------
def _autocast_gpu_worker(rank, world):
    import dear_pytorch_b200 as dear
    dev = dear.device()
    torch.manual_seed(0)
    model = nn.Sequential(nn.Linear(16, 32), nn.ReLU(), nn.Linear(32, 4)).to(dev)
    opt = dear.DistributedOptimizer(torch.optim.SGD(model.parameters(), lr=0.1), model, threshold=0.0001, verbose=False)
    g = torch.Generator().manual_seed(5)
    for _ in range(3):
        x = torch.randn(8, 16, generator=g).to(dev)
        opt.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = model(x).float().pow(2).mean()
        loss.backward()
        opt.step()
    opt.synchronize()
    return [p.detach().float().cpu() for p in model.parameters()]


def test_direct_wgrad_under_cuda_autocast():
    on = run_ranks(_autocast_gpu_worker, world=1, backend="b200", extra_env=ENV, timeout=300)[0]
    off = run_ranks(_autocast_gpu_worker, world=1, backend="b200", extra_env=dict(ENV, DEAR_DIRECT_WGRAD="0"), timeout=300)[0]
    for a, b in zip(on, off):
        torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-6)


# ---- rotated graph body + per-step LR schedule: the deferred update uses the hyper-parameters of its own call ----------------------
def test_rotated_cuda_graph_with_lr_scheduler_and_eager_interruption():
    from test_gpu_fused import check_graph_with_lr_scheduler
    check_graph_with_lr_scheduler(True)


# ---- bench.py: delayed prefetcher uploads (rotated step) --------------------------------------------------------------------
def test_prefetcher_with_delayed_uploads_delivers_every_batch_intact():
    """The copy-stream spin in front of each upload (bench.py's end-to-end run with the rotated step) must not change
    what arrives: 12 batches through a 3-slot ring, each checked against its host original after a consumer kernel."""
    from dear_pytorch_b200.utils.data import PinnedPrefetcher
    dev = torch.device("cuda:0")
    host = [torch.full((1 << 20,), float(i)).pin_memory() for i in range(12)]
    feed = PinnedPrefetcher(iter([(h,) for h in host]), dev, upload_delay_us=300.0)
    if feed._delay_cycles == 0:
        pytest.skip("torch.cuda._sleep is not usable in this build: the prefetcher runs without the delay")
    sums = []
    for (x,) in feed:
        sums.append(x.double().sum())              # consumer work on the current stream
    torch.cuda.synchronize()
    assert [float(s) for s in sums] == [float(i) * (1 << 20) for i in range(12)]


# ---- NCCL-style baselines through the command-line driver (own process group of the ByteScheduler thread, Horovod options) ---------
def _driver_gpu_worker(rank, world, method, extra):
    import contextlib
    import io
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "benchmarks"))
    import imagenet_benchmark as drv
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        res = drv.main(["--model", "resnet18", "--image-size", "64", "--batch-size", "4", "--num-warmup-batches", "2",
                        "--num-batches-per-iter", "2", "--num-iters", "2", "--method", method] + list(extra))
    return res["total"], buf.getvalue()


@pytest.mark.parametrize("method,extra", [("bytescheduler", ()), ("horovod", ()), ("horovod", ("--fp16-allreduce",)),
                                          ("horovod", ("--use-adasum",))])
def test_baseline_methods_of_the_driver_over_nccl(method, extra):
    if torch.cuda.device_count() < 2:
        pytest.skip("NCCL needs one GPU per rank")
    outs = run_ranks(_driver_gpu_worker, world=2, backend="nccl", args=(method, extra), extra_env=ENV, timeout=600)
    total, text = outs[0]
    assert total > 0 and "Total img/sec on 2 GPU(s): " in text


# ---- a slice of the randomised equivalence fuzzer on the fused kernels -----------------------------------------------------------
def test_fuzz_slice_on_the_fused_kernels(monkeypatch):
    """tools/fuzz_equivalence.py with ``--backends b200``: random models / optimizers / bucketing / accumulation / re-bucketing /
    state-dict round trips / TrainStep bodies on the GPU data path against single-process torch.optim on the CPU."""
    import importlib
    import os
    # CUDA ranks are spawned, not forked: they unpickle the fuzzer's worker by module name, so the module must be
    # importable under its own name from a path the children inherit
    monkeypatch.syspath_prepend(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    fuzz = importlib.import_module("fuzz_equivalence")
    failures = fuzz.main(["--seed", "5", "--trials", "6", "--backends", "b200", "--max-world", "2", "--quiet",
                          "--variants", "dear,dear,dear,bo,naive,wt,rb"])
    assert not failures, failures[0]
