"""Every dispatched variant of the communication kernels against a float64 reference of the same operation.

Kernel A (reduce-scatter: one-shot ``rs_kernel`` and stripe-pipelined ``rs_pipe_kernel``), Kernel B (update +
all-gather, SGD and Adam) and ``gen_kernel`` (the standalone collectives) each pick a template instance per dtype
(fp32 / bf16 / fp16) and per world size (1, 2, 4, 8 and a generic instance for every other world, e.g. 3).  This file
runs each instance, at the edges where such kernels go wrong: odd sizes and vector tails, zero-filled and in-place
segments, sums that overflow or cancel in 16-bit arithmetic, non-finite gradients, a gradient scale, host-side
chunking through the staging slot and tensor views that are not 16-byte aligned.

Every reference is computed in float64 from the exact values the kernel saw (after rounding to the storage dtype).
Each case runs on the host emulation (CPU) and, with the gpu marker, on the CUDA kernels, with the same assertions."""
import pytest
import torch
import torch.nn as nn

from _mp import run_ranks
from test_kernels_direct import PIPE_ENV, reference_update

TORCH_DTYPE = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
NATIVE_DTYPE = {"fp32": "DT_F32", "bf16": "DT_BF16", "fp16": "DT_F16"}
U32 = 2.0 ** -24                     # unit roundoff of float32

BACKENDS = ["emu", pytest.param("b200", marks=pytest.mark.gpu)]
GPU_ENV = {"DEAR_SPIN_TIMEOUT_S": "15"}
# the same variables on both backends, so that an emulation case and its CUDA twin run the same plan
ALGO_ENV = {"oneshot": GPU_ENV, "pipe": PIPE_ENV}


def _run(fn, world, backend, args, env):
    _skip_unless_fits(backend, world, env)
    return run_ranks(fn, world=world, backend=backend, args=(backend == "b200",) + tuple(args), extra_env=env,
                     timeout=300 if backend == "b200" else 240)


def _skip_unless_fits(backend, world, env):
    """The one-shot kernels: 2-4 ranks may share one GPU, otherwise every rank needs its own.  The stripe-pipelined
    kernel, like test_kernels_direct's pipelined case: at most 2 ranks may share one GPU."""
    if backend != "b200":
        return
    ngpu = torch.cuda.device_count()
    share = 2 if env.get("DEAR_RS_ALGO") == "pipe" else 4
    if ngpu < world and not (ngpu == 1 and world <= share):
        pytest.skip("the %d-rank case needs %d GPUs" % (world, world))


# ---------------------------------------------------------------------------------------------------------------------
# comparison helpers
# ---------------------------------------------------------------------------------------------------------------------
def ulp_distance(a, b):
    """Number of representable values of the (common) floating dtype between ``a`` and ``b``, elementwise."""
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    ity, mag = (torch.int32, 0x7FFFFFFF) if a.dtype == torch.float32 else (torch.int16, 0x7FFF)

    def key(t):                     # sign-magnitude bit pattern -> monotonic integer (+0 and -0 both map to 0)
        i = t.contiguous().view(ity).to(torch.int64)
        return torch.where(i < 0, -(i & mag), i)
    return (key(a.cpu()) - key(b.cpu())).abs()


def assert_fp32_sum(got, ref, abs_sum, nterms, what):
    """``got`` (float32) is a sum of ``nterms`` terms accumulated in float32 and then scaled once.  Recursive summation
    errs by at most (nterms-1)*u*sum|x|; the scale and its float32 rounding add 2*u*|result|.  ``ref`` and
    ``abs_sum`` are float64 and already scaled."""
    assert got.dtype == torch.float32, got.dtype
    got = got.cpu().double()
    tol = (nterms + 2) * U32 * abs_sum
    bad = ~((got - ref).abs() <= tol)
    if bad.any():
        i = int(bad.nonzero()[0, 0])
        raise AssertionError("%s: %d of %d elements off the float64 reference, first at %d: got %r want %r (tol %.3g)"
                             % (what, int(bad.sum()), got.numel(), i, float(got[i]), float(ref[i]), float(tol[i])))


def assert_ulps(got, want, max_ulps, what):
    d = ulp_distance(got, want)
    if d.numel() and int(d.max()) > max_ulps:
        i = int(d.argmax())
        raise AssertionError("%s: %d elements more than %d ulp off, worst at %d: got %r want %r (%d ulp)"
                             % (what, int((d > max_ulps).sum()), max_ulps, i, float(got.flatten()[i]),
                                float(want.flatten()[i]), int(d[i])))


def assert_reduced(got, sum64, abs64, scale, nterms, what):
    """A reduction returned in the element type: float32 within the float32 summation bound; a 16-bit type within
    1 ulp of the float64 result rounded once to that type."""
    ref = sum64 * scale
    if got.dtype == torch.float32:
        assert_fp32_sum(got, ref, abs64 * abs(scale), nterms, what)
    else:
        assert_ulps(got.cpu(), ref.to(got.dtype), 1, what)


def _layout(numels, es, world):
    """Parameter starts 256-byte aligned like the bucket planner; padded so each shard is a whole number of vectors."""
    align = 256 // es
    starts, off = [], 0
    for n in numels:
        off = (off + align - 1) // align * align
        starts.append(off)
        off += n
    quantum = world * (128 // es)
    return starts, (off + quantum - 1) // quantum * quantum


# ---------------------------------------------------------------------------------------------------------------------
# 1. Kernel A + B: dtype x world x algorithm
# ---------------------------------------------------------------------------------------------------------------------
def matrix_worker(rank, world, use_cuda, dtype_name, seed):
    """Three SGD steps through BucketSet.reduce_scatter + allgather_update: odd parameter sizes, a zero-filled and an
    in-place segment, three hyper-parameter segments (momentum, nesterov + weight decay, plain SGD)."""
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200 import ops
    C = ops.require_native()
    comm = dear.communicator()
    dev = dear.device()
    tdt = TORCH_DTYPE[dtype_name]
    es = torch.tensor([], dtype=tdt).element_size()
    numels = [37, 1000, 4099, 3, 70001]
    starts, padded = _layout(numels, es, world)
    shard = padded // world
    lo, hi = rank * shard, (rank + 1) * shard
    bs = C.BucketSet(comm, [padded], getattr(C, NATIVE_DTYPE[dtype_name]), True)
    pbuf, gbuf = bs.param_buffer(0), bs.grad_buffer(0)
    g = torch.Generator().manual_seed(seed)
    full_p = torch.zeros(padded)
    for s, n in zip(starts, numels):
        full_p[s:s + n] = torch.randn(n, generator=g)
    pbuf.copy_(full_p.to(tdt))
    ref_p = pbuf.cpu().double()                                  # what the kernel starts from
    gs = torch.zeros(shard, device=dev)
    mom = torch.zeros(shard, device=dev)
    master = pbuf[lo:hi].float().clone() if tdt != torch.float32 else None
    bs.set_shards(0, gs, mom, master)
    hyp = [(starts[2], 0.1, 0.01, 0.9, 0.0, 0), (starts[4], 0.05, 0.0, 0.8, 0.0, 1), (padded, 0.2, 0.001, 0.0, 0.0, 0)]
    bs.set_hyper(0, [h[0] for h in hyp], [h[1] for h in hyp], [h[2] for h in hyp], [h[3] for h in hyp],
                 [h[4] for h in hyp], [h[5] for h in hyp])
    ref_buf = torch.zeros(padded, dtype=torch.float64)
    buckets = []
    for step in range(3):
        # param 3 is absent on step 1 (zero fill), param 1 is already in the bucket on step 2
        gen = torch.Generator().manual_seed(1000 * step + 7)
        all_rank_grads = [[torch.randn(n, generator=gen).to(tdt) for n in numels] for _ in range(world)]
        mine = [t.to(dev) for t in all_rank_grads[rank]]
        src, flags = [], []
        for i, t in enumerate(mine):
            if step == 1 and i == 3:
                src.append(0); flags.append(C.SEG_ZERO_FILL)
            elif step == 2 and i == 1:
                gbuf[starts[i]:starts[i] + numels[i]].copy_(t)
                src.append(0); flags.append(0)
            else:
                src.append(t.data_ptr()); flags.append(0)
        bs.set_pack(0, src, [s * es for s in starts], [n * es for n in numels], flags)
        bs.reduce_scatter(0, True)
        bs.allgather_update(0, True, step == 0, True, False)
        bs.synchronize()
        comm.check_status()

        summed = torch.zeros(padded, dtype=torch.float64)
        abs_sum = torch.zeros(padded, dtype=torch.float64)
        for r in range(world):
            for i, (s, n) in enumerate(zip(starts, numels)):
                if not (step == 1 and i == 3):
                    summed[s:s + n] += all_rank_grads[r][i].double()
                    abs_sum[s:s + n] += all_rank_grads[r][i].double().abs()
        avg = summed / world
        start = 0
        for end, lr, wd, m, damp, nest in hyp:
            sl = slice(start, end)
            ref_p[sl], ref_buf[sl] = reference_update(ref_p[sl], avg[sl], ref_buf[sl], step == 0, lr, wd, m, damp, bool(nest))
            start = end
        what = "step %d rank %d" % (step, rank)
        assert_fp32_sum(gs, avg[lo:hi], abs_sum[lo:hi] / world, world, what + " reduced shard")
        bucket = pbuf.cpu().clone()
        if tdt == torch.float32:
            torch.testing.assert_close(bucket.double(), ref_p, rtol=1e-5, atol=1e-6, msg=what + " parameters")
        else:
            torch.testing.assert_close(master.cpu().double(), ref_p[lo:hi], rtol=1e-5, atol=1e-6, msg=what + " master")
            # the bucket is the fp32 master rounded once to nearest: bit-exact on my shard, <= 1 ulp from float64
            assert_ulps(bucket[lo:hi], master.cpu().to(tdt), 0, what + " bucket vs master")
            assert_ulps(bucket, ref_p.to(tdt), 1, what + " bucket vs float64 reference")
        buckets.append(bucket)
    return buckets


# world 1 always runs the one-shot kernel (there is nothing to pipeline), so "pipe" starts at 2 ranks
MATRIX = [(w, a) for w in (1, 2, 3, 4, 8) for a in ("oneshot", "pipe") if not (w == 1 and a == "pipe")]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("dtype_name", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("world,algo", MATRIX)
def test_sgd_kernels_match_float64(world, algo, dtype_name, backend):
    outs = _run(matrix_worker, world, backend, (dtype_name, 5), ALGO_ENV[algo])
    for r in range(1, world):
        for a, b in zip(outs[0], outs[r]):
            assert torch.equal(a, b), "rank %d holds a different bucket than rank 0" % r


def adam_worker(rank, world, use_cuda, dtype_name, seed):
    """Kernel B with the Adam / AdamW epilogue against torch.optim.Adam(W) in float64 on the averaged gradient."""
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200 import ops
    C = ops.require_native()
    comm = dear.communicator()
    dev = dear.device()
    tdt = TORCH_DTYPE[dtype_name]
    es = torch.tensor([], dtype=tdt).element_size()
    numels = [513, 4099, 70001]
    starts, padded = _layout(numels, es, world)
    shard = padded // world
    lo, hi = rank * shard, (rank + 1) * shard
    bs = C.BucketSet(comm, [padded], getattr(C, NATIVE_DTYPE[dtype_name]), True)
    pbuf = bs.param_buffer(0)
    g = torch.Generator().manual_seed(seed)
    full_p = torch.zeros(padded)
    for s, n in zip(starts, numels):
        full_p[s:s + n] = torch.randn(n, generator=g)
    pbuf.copy_(full_p.to(tdt))
    full_p = pbuf.cpu().double()
    gs = torch.zeros(shard, device=dev)
    m = torch.zeros(shard, device=dev)
    v = torch.zeros(shard, device=dev)
    master = pbuf[lo:hi].float().clone() if tdt != torch.float32 else None
    bs.set_shards(0, gs, m, master, v)
    bs.set_step(0, 0)
    # params 0-1: Adam with L2 weight decay; param 2: AdamW
    hyp = [(starts[2], 1e-2, 1e-2, 0.9, 0.999, 1e-8, C.OPT_ADAM), (padded, 5e-3, 5e-2, 0.8, 0.95, 1e-6, C.OPT_ADAMW)]
    bs.set_hyper(0, [h[0] for h in hyp], [h[1] for h in hyp], [h[2] for h in hyp], [h[3] for h in hyp],
                 [0.0] * len(hyp), [0] * len(hyp), opt=[h[6] for h in hyp], beta2=[h[4] for h in hyp], eps=[h[5] for h in hyp])
    ref_params = [torch.nn.Parameter(full_p[s:s + n].clone()) for s, n in zip(starts, numels)]
    ref_opts = [torch.optim.Adam(ref_params[:2], lr=1e-2, weight_decay=1e-2, betas=(0.9, 0.999), eps=1e-8),
                torch.optim.AdamW(ref_params[2:], lr=5e-3, weight_decay=5e-2, betas=(0.8, 0.95), eps=1e-6)]
    buckets = []
    for step in range(4):
        gen = torch.Generator().manual_seed(1000 * step + 11)
        all_rank_grads = [[torch.randn(n, generator=gen).to(tdt) for n in numels] for _ in range(world)]
        mine = [t.to(dev) for t in all_rank_grads[rank]]
        bs.set_pack(0, [t.data_ptr() for t in mine], [s * es for s in starts], [n * es for n in numels], [0] * len(numels))
        bs.reduce_scatter(0, True)
        bs.allgather_update(0, True, step == 0, True, False)
        bs.synchronize()
        comm.check_status()
        for i, p in enumerate(ref_params):
            p.grad = sum(all_rank_grads[r][i].double() for r in range(world)) / world
        for o in ref_opts:
            o.step()
        ref = torch.zeros(padded, dtype=torch.float64)
        for s, n, p in zip(starts, numels, ref_params):
            ref[s:s + n] = p.detach()
        what = "step %d rank %d" % (step, rank)
        bucket = pbuf.cpu().clone()
        if tdt == torch.float32:
            torch.testing.assert_close(bucket.double(), ref, rtol=2e-5, atol=2e-6, msg=what + " parameters")
        else:
            torch.testing.assert_close(master.cpu().double(), ref[lo:hi], rtol=2e-5, atol=2e-6, msg=what + " master")
            assert_ulps(bucket[lo:hi], master.cpu().to(tdt), 0, what + " bucket vs master")
            assert_ulps(bucket, ref.to(tdt), 1, what + " bucket vs float64 reference")
        buckets.append(bucket)
    return buckets


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("world,dtype_name", [(1, "fp16"), (2, "fp16"), (3, "fp16"), (3, "fp32"), (3, "bf16")])
def test_adam_kernel_matches_float64(world, dtype_name, backend):
    outs = _run(adam_worker, world, backend, (dtype_name, 9), GPU_ENV)
    for r in range(1, world):
        for a, b in zip(outs[0], outs[r]):
            assert torch.equal(a, b), "rank %d holds a different bucket than rank 0" % r


# ---------------------------------------------------------------------------------------------------------------------
# 2. accumulation precision and range of Kernel A
# ---------------------------------------------------------------------------------------------------------------------
def _range_grads(case, world, padded):
    """Every rank's gradient bucket for one accumulation case (float64 values exactly representable in the dtype)."""
    i = torch.arange(padded)
    sign = torch.where((i // 5) % 2 == 0, 1.0, -1.0).double()
    if case == "fp16_overflow":
        # the sum of two or more ranks is above the fp16 maximum (65504): a half-precision accumulator gives inf
        return [60000.0 * sign for _ in range(world)]
    if case == "bf16_cancel":
        # 256 + 1 = 257 is not a bf16 number: accumulated in bf16 in rank order the sum is 256 - 256 = 0, in fp32 it is 1
        assert world == 3
        return [256.0 * sign, sign.clone(), -256.0 * sign]
    g = torch.Generator().manual_seed(77)
    grads = [torch.randn(padded, generator=g).double() for _ in range(world)]
    grads[world - 1][5] = float("inf")            # shard 0
    grads[0][padded - 3] = float("-inf")          # last shard
    grads[world // 2][padded // 2 + 6] = float("nan")
    return grads


def range_worker(rank, world, use_cuda, case, dtype_name):
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200 import ops
    C = ops.require_native()
    comm = dear.communicator()
    dev = dear.device()
    tdt = TORCH_DTYPE[dtype_name]
    es = torch.tensor([], dtype=tdt).element_size()
    shard = 4104                                  # not a power of two: the grid-stride loops end on a partial pass
    padded = world * shard
    lo, hi = rank * shard, (rank + 1) * shard
    grads = [t.to(tdt) for t in _range_grads(case, world, padded)]
    bs = C.BucketSet(comm, [padded], getattr(C, NATIVE_DTYPE[dtype_name]), True)
    gs = torch.zeros(shard, device=dev)
    bs.set_shards(0, gs, None, None)
    mine = grads[rank].to(dev)
    bs.set_pack(0, [mine.data_ptr()], [0], [padded * es], [0])
    bs.reduce_scatter(0, True)
    bs.synchronize()
    comm.check_status()
    got = gs.cpu()
    g64 = torch.stack([t.double() for t in grads])
    mean = g64.sum(0)[lo:hi] / world
    what = "%s %s rank %d" % (case, dtype_name, rank)
    if case == "bf16_cancel":
        # exactly the sum (+-1) times the kernel's float32 scale 1/P
        want = (torch.sign(mean) * torch.tensor(1.0 / world, dtype=torch.float32).double()).float()
        assert torch.equal(got, want), "%s: got %s" % (what, got[:8].tolist())
        return got
    finite = torch.isfinite(mean)
    assert torch.equal(torch.isnan(got), torch.isnan(mean)), what + ": NaN in the wrong elements"
    assert torch.equal(torch.isinf(got), torch.isinf(mean)), what + ": inf in the wrong elements"
    assert torch.equal(got[torch.isinf(mean)], mean[torch.isinf(mean)].float()), what + ": wrong sign of inf"
    assert_fp32_sum(got[finite], mean[finite], g64.abs().sum(0)[lo:hi][finite] / world, world, what)
    return got


RANGE_CASES = [("fp16_overflow", "fp16", 2), ("fp16_overflow", "fp16", 3), ("bf16_cancel", "bf16", 3),
               ("nonfinite", "fp32", 3), ("nonfinite", "bf16", 3), ("nonfinite", "fp16", 3), ("nonfinite", "fp16", 2)]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("algo", ["oneshot", "pipe"])
@pytest.mark.parametrize("case,dtype_name,world", RANGE_CASES)
def test_reduce_scatter_accumulates_in_fp32(case, dtype_name, world, algo, backend):
    outs = _run(range_worker, world, backend, (case, dtype_name), ALGO_ENV[algo])
    if case == "nonfinite":
        full = torch.cat(outs)
        assert int(torch.isnan(full).sum()) == 1 and int(torch.isinf(full).sum()) == 2, "a non-finite value spread"


# ---------------------------------------------------------------------------------------------------------------------
# 3. gradient scale (static loss scaling folded into Kernel A)
# ---------------------------------------------------------------------------------------------------------------------
def grad_scale_worker(rank, world, use_cuda, dtype_name):
    """set_grad_scale(0.25): the reduced shard is 0.25 * mean, whether the gradients are packed by the kernel or are
    already in the bucket (on one GPU these are the two branches of the direct pack into the fp32 shard)."""
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200 import ops
    C = ops.require_native()
    comm = dear.communicator()
    dev = dear.device()
    tdt = TORCH_DTYPE[dtype_name]
    es = torch.tensor([], dtype=tdt).element_size()
    numels = [37, 4099, 70001]
    starts, padded = _layout(numels, es, world)
    shard = padded // world
    lo, hi = rank * shard, (rank + 1) * shard
    bs = C.BucketSet(comm, [padded], getattr(C, NATIVE_DTYPE[dtype_name]), True)
    gbuf = bs.grad_buffer(0)
    gs = torch.zeros(shard, device=dev)
    bs.set_shards(0, gs, None, None)
    bs.set_grad_scale(0.25)
    for step, mode in enumerate(["packed", "inplace", "packed"]):
        gen = torch.Generator().manual_seed(500 + step)
        all_rank_grads = [[torch.randn(n, generator=gen).to(tdt) for n in numels] for _ in range(world)]
        mine = [t.to(dev) for t in all_rank_grads[rank]]
        if mode == "inplace":
            for s, t in zip(starts, mine):
                gbuf[s:s + t.numel()].copy_(t)
        src = [t.data_ptr() if mode == "packed" else 0 for t in mine]
        bs.set_pack(0, src, [s * es for s in starts], [n * es for n in numels], [0] * len(numels))
        bs.reduce_scatter(0, True)
        bs.synchronize()
        comm.check_status()
        summed = torch.zeros(padded, dtype=torch.float64)
        abs_sum = torch.zeros(padded, dtype=torch.float64)
        for r in range(world):
            for s, t in zip(starts, all_rank_grads[r]):
                summed[s:s + t.numel()] += t.double()
                abs_sum[s:s + t.numel()] += t.double().abs()
        assert_fp32_sum(gs, summed[lo:hi] / world * 0.25, abs_sum[lo:hi] / world * 0.25, world,
                        "%s step %d rank %d" % (mode, step, rank))
    return True


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("dtype_name", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("world", [1, 2, 3])
def test_grad_scale_applies_to_the_reduced_shard(world, dtype_name, backend):
    _run(grad_scale_worker, world, backend, (dtype_name,), GPU_ENV)


def _conv_net():
    torch.manual_seed(0)
    # no Linear layer: every gradient is packed by Kernel A, so one rank takes the direct pack into the fp32 shard
    return nn.Sequential(nn.Conv2d(3, 8, 3, padding=1), nn.ReLU(), nn.Conv2d(8, 10, 3, padding=1, bias=False),
                         nn.AdaptiveAvgPool2d(1), nn.Flatten())


def loss_scale_worker(rank, world, use_cuda, steps):
    import dear_pytorch_b200 as dear
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cudnn.deterministic = True
    dev = dear.device()
    model, ref = _conv_net().to(dev), _conv_net().to(dev)
    kw = dict(lr=0.05, momentum=0.9, weight_decay=1e-3)
    opt = dear.DistributedOptimizer(torch.optim.SGD(model.parameters(), **kw), model, verbose=False)
    opt.set_loss_scale(64)
    ref_opt = torch.optim.SGD(ref.parameters(), **kw)
    for t in range(steps):
        g = torch.Generator().manual_seed(300 + t)
        x, y = torch.randn(8, 3, 8, 8, generator=g).to(dev), torch.randint(0, 10, (8,), generator=g).to(dev)
        opt.zero_grad()
        (nn.functional.cross_entropy(model(x), y) * 64).backward()
        opt.step()
        ref_opt.zero_grad()
        nn.functional.cross_entropy(ref(x), y).backward()
        ref_opt.step()
    opt.synchronize()
    dear.communicator().check_status()
    return [p.detach().cpu() for p in model.parameters()], [p.detach().cpu() for p in ref.parameters()]


@pytest.mark.parametrize("backend", BACKENDS)
def test_loss_scale_on_one_rank_matches_unscaled_sgd(backend):
    (got, want), = _run(loss_scale_worker, 1, backend, (3,), GPU_ENV)
    for a, b in zip(got, want):
        torch.testing.assert_close(a, b, rtol=0, atol=1e-5)


# ---------------------------------------------------------------------------------------------------------------------
# 4. general collectives (gen_kernel)
# ---------------------------------------------------------------------------------------------------------------------
STAGING_MB = 1


def gen_worker(rank, world, use_cuda, dtype_name):
    """allReduce, reduce, bcast, reduceScatter, allGather, sendrecv, allReduceRSAG and allReduceRB on whole tensors of
    1, 7, 4099 and more than twice the staging slot's elements, plus views one element off an aligned allocation."""
    import dear_pytorch_b200 as dear
    comm = dear.communicator()
    dev = dear.device()
    tdt = TORCH_DTYPE[dtype_name]
    es = torch.tensor([], dtype=tdt).element_size()
    slot = (STAGING_MB << 20) // es
    big = (2 * slot + 4099 + 11) // 12 * 12       # > 2 staging slots; divisible by 2, 3 and 4 so RSAG does not fall back
    last = world - 1
    inv = 1.0 / world

    def x(n, r, salt=0):
        g = torch.Generator().manual_seed(100003 * salt + 1009 * r + n)
        return torch.randn(n, generator=g).to(tdt)

    def sync(h):
        comm.syncStream(h)

    def stats(ts):
        t64 = torch.stack([t.double() for t in ts])
        return t64.sum(0), t64.abs().sum(0)

    for n in (1, 7, 4099, big):
        xs = [x(n, r) for r in range(world)]
        s64, a64 = stats(xs)
        what = lambda op: "%s n=%d rank %d" % (op, n, rank)   # noqa: E731

        t = xs[rank].to(dev, copy=True)
        sync(comm.allReduce(t, inv))
        assert_reduced(t, s64, a64, inv, world, what("allReduce"))

        t = xs[rank].to(dev, copy=True)
        sync(comm.reduce(t, last, 1.0))
        if rank == last:
            assert_reduced(t, s64, a64, 1.0, world, what("reduce"))
        else:
            assert torch.equal(t.cpu(), xs[rank]), what("reduce") + ": a non-root tensor changed"

        t = xs[rank].to(dev, copy=True)
        sync(comm.bcast(t, last))
        assert torch.equal(t.cpu(), xs[last]), what("bcast")
        gi = torch.Generator().manual_seed(n + rank)
        ints = torch.randint(-2 ** 62, 2 ** 62, (n,), generator=gi, dtype=torch.int64)
        gi = torch.Generator().manual_seed(n + last)
        root_ints = torch.randint(-2 ** 62, 2 ** 62, (n,), generator=gi, dtype=torch.int64)
        t = ints.to(dev, copy=True)
        sync(comm.bcast(t, last))
        assert torch.equal(t.cpu(), root_ints), what("bcast int64")

        sends = [x(world * n, r, 1) for r in range(world)]
        rs64, ra64 = stats([s[rank * n:(rank + 1) * n] for s in sends])
        send, recv = sends[rank].to(dev, copy=True), torch.empty(n, dtype=tdt, device=dev)
        sync(comm.reduceScatter(send, recv, inv))
        assert_reduced(recv, rs64, ra64, inv, world, what("reduceScatter"))

        send, recv = xs[rank].to(dev, copy=True), torch.empty(world * n, dtype=tdt, device=dev)
        sync(comm.allGather(send, recv))
        assert torch.equal(recv.cpu(), torch.cat(xs)), what("allGather")

        send, recv = xs[rank].to(dev, copy=True), torch.empty(n, dtype=tdt, device=dev)
        sync(comm.sendrecv(send, recv, (rank + 1) % world))
        assert torch.equal(recv.cpu(), xs[(rank + 1) % world]), what("sendrecv")

        t = xs[rank].to(dev, copy=True)
        sync(comm.allReduceRSAG(t, inv))
        assert_reduced(t, s64, a64, inv, world, what("allReduceRSAG"))

        t = xs[rank].to(dev, copy=True)
        sync(comm.allReduceRB(t, inv))
        assert_reduced(t, s64, a64, inv, world, what("allReduceRB"))

    # views one element past an aligned allocation: 4-byte (fp32, int64 is 8) or 2-byte (16-bit) aligned pointers.
    # The element in front of each view must survive.
    for n in (7, 4099):
        xs = [x(n, r, 2) for r in range(world)]
        s64, a64 = stats(xs)
        what = lambda op: "%s on a misaligned view, n=%d rank %d" % (op, n, rank)   # noqa: E731

        def view_of(t, fill=-3.0):
            buf = torch.full((t.numel() + 1,), fill, dtype=t.dtype, device=dev)
            buf[1:].copy_(t)
            return buf

        buf = view_of(xs[rank])
        sync(comm.allReduce(buf[1:], inv))
        assert_reduced(buf[1:], s64, a64, inv, world, what("allReduce"))
        assert float(buf[0]) == -3.0, what("allReduce") + ": wrote in front of the view"

        buf = view_of(xs[rank])
        sync(comm.reduce(buf[1:], last, 1.0))
        if rank == last:
            assert_reduced(buf[1:], s64, a64, 1.0, world, what("reduce"))
        assert float(buf[0]) == -3.0, what("reduce") + ": wrote in front of the view"

        buf = view_of(xs[rank])
        sync(comm.bcast(buf[1:], last))
        assert torch.equal(buf.cpu(), torch.cat([torch.tensor([-3.0], dtype=tdt), xs[last]])), what("bcast")

        ibuf = torch.full((n + 1,), -7, dtype=torch.int64, device=dev)
        ibuf[1:] = torch.arange(n, device=dev) * 1000003 + rank
        sync(comm.bcast(ibuf[1:], last))
        assert int(ibuf[0]) == -7 and torch.equal(ibuf[1:].cpu(), torch.arange(n) * 1000003 + last), what("bcast int64")

        sbuf, rbuf = view_of(xs[rank]), torch.full((world * n + 1,), -3.0, dtype=tdt, device=dev)
        sync(comm.allGather(sbuf[1:], rbuf[1:]))
        assert float(rbuf[0]) == -3.0 and torch.equal(rbuf[1:].cpu(), torch.cat(xs)), what("allGather")

        sbuf, rbuf = view_of(xs[rank]), torch.full((n + 1,), -3.0, dtype=tdt, device=dev)
        sync(comm.sendrecv(sbuf[1:], rbuf[1:], (rank + 1) % world))
        assert float(rbuf[0]) == -3.0 and torch.equal(rbuf[1:].cpu(), xs[(rank + 1) % world]), what("sendrecv")

    comm.check_status()
    return True


GEN_CASES = [(2, "fp32"), (2, "bf16"), (2, "fp16"), (3, "fp32"), (3, "bf16"), (3, "fp16"), (4, "fp32"), (4, "bf16"),
             (4, "fp16")]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("world,dtype_name", GEN_CASES)
def test_general_collectives_match_float64(world, dtype_name, backend):
    env = dict(GPU_ENV, DEAR_STAGING_MB=str(STAGING_MB))      # several chunks through the staging slot
    _run(gen_worker, world, backend, (dtype_name,), env)


# ---------------------------------------------------------------------------------------------------------------------
# 5. the emulation and the CUDA kernels agree bit for bit
# ---------------------------------------------------------------------------------------------------------------------
def shard_worker(rank, world, use_cuda, seed):
    """One fp32 reduce-scatter of seeded gradients; returns this rank's reduced shard."""
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200 import ops
    C = ops.require_native()
    comm = dear.communicator()
    dev = dear.device()
    numels = [37, 4099, 70001]
    starts, padded = _layout(numels, 4, world)
    bs = C.BucketSet(comm, [padded], C.DT_F32, True)
    gs = torch.zeros(padded // world, device=dev)
    bs.set_shards(0, gs, None, None)
    gen = torch.Generator().manual_seed(seed)
    grads = [[torch.randn(n, generator=gen) for n in numels] for _ in range(world)]
    mine = [t.to(dev) for t in grads[rank]]
    bs.set_pack(0, [t.data_ptr() for t in mine], [s * 4 for s in starts], [n * 4 for n in numels], [0] * len(numels))
    bs.reduce_scatter(0, True)
    bs.synchronize()
    comm.check_status()
    return gs.cpu()


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["oneshot", "pipe"])
@pytest.mark.parametrize("world", [2, 3])
def test_emulation_and_cuda_reduce_scatter_are_bit_identical(world, algo):
    """Both sum the ranks in the same fixed order in float32 and then multiply by the same float32 1/P."""
    env = ALGO_ENV[algo]
    emu = torch.cat(_run(shard_worker, world, "emu", (21,), env))
    cuda = torch.cat(_run(shard_worker, world, "b200", (21,), env))
    assert torch.equal(emu, cuda), "max ulp difference %d" % int(ulp_distance(emu, cuda).max())
