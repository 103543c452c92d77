#!/usr/bin/env python
"""Headline benchmark: ResNet-50, batch 64 per GPU, synthetic ImageNet, DeAR with tensor fusion.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, 1 rank/GPU)
    python bench.py --impl reference ...                     (the reference's own code path over NCCL)
    python bench.py --model bert --dtype bf16 ...            (BERT-large pre-training, samples/s)

Metric and config follow BASELINE.json ("ResNet-50 images/sec ... bs=64/GPU synthetic ImageNet
DeAR-TF", "BERT-large pretraining bf16 DeAR-TF") and the reference drivers
dear/imagenet_benchmark.py / dear/bert_benchmark.py (SGD, synthetic batch, cross-entropy).
Timing: W untimed warm-up steps, then exactly K steps between CUDA events, bracketed by
barrier + synchronize, max over ranks.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BASELINE_PUBLISHED = None   # the reference publishes no throughput number (BASELINE.md §1)
BERT_MODELS = ("bert", "bert_large", "bert_base")
DUMP_STATE_SAMPLE = 1 << 22      # --dump-outputs: 16 MB of float32; >= 1 % of BERT-large's 336 M elements


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["dear", "reference"], default="dear")
    ap.add_argument("--model", default="resnet50")
    ap.add_argument("--batch-size", type=int, default=None, help="per GPU (default: 64 images / 32 sentences)")
    ap.add_argument("--sentence-len", type=int, default=64)
    ap.add_argument("--dtype", choices=["fp32", "bf16", "amp"], default=os.environ.get("DEAR_BENCH_DTYPE"))
    ap.add_argument("--channels-last", type=int, default=int(os.environ.get("DEAR_BENCH_CL", "1")))
    ap.add_argument("--graph", type=int, default=int(os.environ.get("DEAR_BENCH_GRAPH", "1")),
                    help="replay the whole iteration as one CUDA graph (GPU only; validated at 1/2/8 GPUs)")
    ap.add_argument("--overlap-update", type=int, default=(int(os.environ["DEAR_BENCH_OVERLAP"]) if "DEAR_BENCH_OVERLAP" in os.environ else None),
                    help="graph mode: capture step(previous gradients) -> forward -> backward so the update + all-gather "
                         "kernels overlap the forward inside the graph (utils/train.py) -- DeAR's defining overlap; default: on "
                         "with peers and for BERT (+3.5 %% on one B200), off for a CNN on a single GPU (nothing to hide; "
                         "the natural body measured faster there)")
    ap.add_argument("--fused-bn", type=int, default=int(os.environ.get("DEAR_BENCH_FUSED_BN", "1")),
                    help="ResNets: fused channels-last BatchNorm(+add)+ReLU kernels (csrc/bn_act.cu)")
    ap.add_argument("--fused-ln", type=int, default=int(os.environ.get("DEAR_BENCH_FUSED_LN", "1")),
                    help="BERT: dropout + add + LayerNorm in one kernel (csrc/ln_fused.cu)")
    ap.add_argument("--tc-ffn", type=int, default=int(os.environ.get("DEAR_BENCH_TC_FFN", "0")),
                    help="BERT bf16: feed-forward block on the hand-written tcgen05 GEMMs with fused GELU epilogues (csrc/tc_ffn_hw.cu); "
                         "off by default: cuBLAS + the fused bias/GELU kernels are faster (profiles/README.md R2.5)")
    ap.add_argument("--threshold", type=float, default=25.0)
    ap.add_argument("--momentum", type=float, default=0.0)
    ap.add_argument("--optimizer", choices=["sgd", "adam", "adamw"], default="sgd",
                    help="sgd = the reference's benchmark optimizer; adam/adamw use the sharded Adam epilogue of Kernel B")
    ap.add_argument("--backend", default=None)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--upload-delay-us", type=float, default=None,
                    help="end-to-end run: spin this long on the copy stream before each prefetch upload so the PCIe DMA does "
                         "not start at the step boundary, where the rotated step runs the update + all-gather kernels "
                         "(utils/data.py). Default: 2000 with --overlap-update 1, else 0")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed (rank 0) as float32 .npy files: "
                         "loss.npy, and model_state.npy, the floating-point entries of the model's state_dict with that "
                         "step's update applied, flattened in state_dict order (a fixed sample of %d elements when larger)"
                         % DUMP_STATE_SAMPLE)
    args = ap.parse_args(argv)
    if args.dump_outputs and (args.impl != "dear" or args.steps < 1):
        ap.error("--dump-outputs needs --impl dear and --steps >= 1")
    is_bert = args.model in BERT_MODELS
    if args.batch_size is None:
        args.batch_size = 32 if is_bert else 64
    if args.dtype is None:
        # BERT-large is specified in bf16 (BASELINE.json); ResNet-50 runs at the reference's precision
        args.dtype = "bf16" if is_bert else "fp32"
    if args.overlap_update is None:
        # Rotated body wherever it measured faster: with peers (it hides the all-gather tail: ResNet-50 13.51 -> 13.38 ms
        # at 8 GPUs) and for BERT even on one GPU (+3.5 %).  A CNN on ONE GPU has no communication to hide and the
        # natural body is faster there (ResNet-50 13.25 vs 13.27 ms resident, 13.26 vs 13.44 ms end to end; VGG-16
        # 21.12 (round-1 eager loop, natural order) vs 21.45 ms), so that case keeps it.
        args.overlap_update = 1 if (is_bert or int(os.environ.get("WORLD_SIZE", "1")) > 1) else 0
    return args


def _free_port():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def main(argv=None):
    args = parse_args(argv)
    if args.gpus > 1 and "RANK" not in os.environ:
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), os.path.abspath(__file__)] + \
              (argv if argv is not None else sys.argv[1:])
        sys.exit(subprocess.call(cmd))
    if args.impl == "reference":
        from baseline.run_reference import run as run_reference
        return run_reference(args)
    return run_dear(args)


class Workload:
    """Model + synthetic data of one benchmark task."""

    def __init__(self, args, device, rank):
        import torch
        import torch.nn.functional as F
        from dear_pytorch_b200.models.registry import create, input_size
        self.args = args
        self.is_bert = args.model in BERT_MODELS
        cuda = device.type == "cuda"
        B = args.batch_size
        if self.is_bert:
            from dear_pytorch_b200.models import bert as bm
            self.fused_ln = bool(args.fused_ln) and cuda
            self.tc_ffn = bool(args.tc_ffn) and cuda and args.dtype == "bf16"
            model = create(args.model, fused_ln=self.fused_ln, tc_ffn=self.tc_ffn).to(device)
            if args.dtype == "bf16":
                model = model.to(torch.bfloat16)
            crit = bm.BertPretrainingCriterion(model.vocab_size)
            self.loss_fn = lambda out, tgt: crit(out[0], out[1], tgt[0], tgt[1])
            self.unit, self.metric = "samples/s", "samples/sec (BERT-%s pre-training, seq %d, DeAR tensor fusion)" % (
                "base" if args.model == "bert_base" else "large", args.sentence_len)

            def host_batch(seed):
                ids, mask, types, nsp, mlm = bm.synthetic_batch(B, args.sentence_len, model.vocab_size, "cpu", seed)
                ts = (ids, types, mask, mlm, nsp)
                return tuple(t.pin_memory() if cuda else t for t in ts)
            self.host_batches = [host_batch(100 * rank + i) for i in range(4)]
            self.to_step_args = lambda b: (b[0], b[1], b[2], (b[3], b[4]))
            self.image = None
        else:
            kw = {"fused_bn": True} if (args.fused_bn and args.channels_last and args.model.startswith(("resnet", "densenet"))) else {}
            model = create(args.model, **kw).to(device)
            self.fused_bn = bool(kw)
            if args.channels_last:
                model = model.to(memory_format=torch.channels_last)
            if args.dtype == "bf16":
                # bf16 parameters / activations / gradients, fp32 BatchNorm; fp32 master weights and
                # momentum live (sharded) inside the optimizer
                model = model.to(torch.bfloat16)
                for m in model.modules():
                    if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
                        m.float()
            self.loss_fn = lambda out, y: F.cross_entropy(out.float() if out.dtype != torch.float32 else out, y)
            self.unit = "images/s"
            self.metric = "images/sec (ResNet-50 synthetic ImageNet training, DeAR tensor fusion)" \
                if args.model == "resnet50" else "images/sec (%s synthetic training, DeAR tensor fusion)" % args.model
            size = input_size(args.model)
            self.image = size
            xdt = torch.bfloat16 if args.dtype == "bf16" else torch.float32
            g = torch.Generator().manual_seed(1000 + rank)

            def host_batch():
                x = torch.randn(B, 3, size, size, generator=g).to(xdt)
                if args.channels_last:
                    x = x.contiguous(memory_format=torch.channels_last)
                y = torch.randint(0, 1000, (B,), generator=g)
                return (x.pin_memory(), y.pin_memory()) if cuda else (x, y)
            self.host_batches = [host_batch() for _ in range(4)]
            self.to_step_args = lambda b: b
        model.train()
        self.model = model
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.host_batches[0])


def run_dear(args):
    import torch
    import dear_pytorch_b200 as dear
    from dear_pytorch_b200.utils.clocks import ClockSampler
    from dear_pytorch_b200.utils.data import PinnedPrefetcher
    from dear_pytorch_b200.utils.train import TrainStep

    dear.init(backend=args.backend)
    rank, world = dear.rank(), dear.size()
    device = dear.device()
    cuda = device.type == "cuda"
    torch.backends.cudnn.benchmark = True
    torch.manual_seed(1234)

    wl = Workload(args, device, rank)
    model = wl.model
    lr = (2e-5 if wl.is_bert else 0.01 * world)          # dear/bert_benchmark.py:122, dear/imagenet_benchmark.py:94
    if args.optimizer == "sgd":
        base = torch.optim.SGD(model.parameters(), lr=lr, momentum=args.momentum)
    else:
        lr *= 0.1
        base = (torch.optim.AdamW if args.optimizer == "adamw" else torch.optim.Adam)(model.parameters(), lr=lr)
    opt = dear.DistributedOptimizer(base, model, threshold=args.threshold,
                                    verbose=(rank == 0 and bool(os.environ.get("DEAR_VERBOSE"))))
    dear.broadcast_parameters(model.state_dict(), 0)
    step = TrainStep(model, opt, wl.loss_fn, autocast_dtype=torch.bfloat16 if args.dtype == "amp" else None,
                     use_graph=bool(args.graph) and cuda, overlap_update=bool(args.overlap_update) and bool(args.graph) and cuda)
    B = args.batch_size

    # ---- device-resident synthetic batch (the reference's protocol) -------------------------
    dev_batch = wl.to_step_args(tuple(t.to(device) for t in wl.host_batches[0]))

    def sync():
        if cuda:
            torch.cuda.synchronize(device)

    comm = dear.communicator()
    from dear_pytorch_b200 import ops as _ops

    def n_launches():
        """kernels of THIS repo launched so far: fused RS / SGD+AG / general collectives + fused BN"""
        n = comm.launches() if comm is not None else opt.engine.backend.launches()
        C = _ops.native()
        if C is not None:
            n += C.bn_act_launches() + C.ln_launches()
        from dear_pytorch_b200.ops.tc_gemm import tc_launches
        return n + tc_launches()

    l_warm = n_launches()
    # W untimed warm-up steps.  In graph mode the capture (3 eager iterations + 1 capturing call) must
    # be over before the timed region starts, whatever W the caller asked for.
    n_warm = max(args.warmup, step.graph_warmup + 2) if step.use_graph else args.warmup
    for _ in range(n_warm):
        step(*dev_batch)
    opt.engine.synchronize(host=True)
    # launches per iteration, counted while the Python step body ran (a replayed CUDA graph launches
    # the same kernels without passing through the host-side counters)
    per_step_launches = (n_launches() - l_warm) / max(1, step.eager_calls)

    def timed(run_one, n):
        dear.barrier(); sync()
        l0 = n_launches()
        if cuda:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        t0 = time.perf_counter()
        for _ in range(n):
            run_one()
        opt.engine.synchronize(host=False)       # the K-th update must have landed
        if cuda:
            e1.record()
            sync()
            ms = e0.elapsed_time(e1)
        else:
            ms = (time.perf_counter() - t0) * 1e3
        dear.barrier()
        return ms, n_launches() - l0

    last_loss = [None]

    def resident():
        last_loss[0] = step(*dev_batch)

    sampler = ClockSampler(device.index if cuda else 0).start() if (cuda and rank == 0) else None
    wall0 = time.time()
    ms, launches = timed(resident, args.steps)
    wall1 = time.time()
    if args.graph and cuda:
        launches = int(round(per_step_launches * args.steps))
    if args.dump_outputs:
        _dump_outputs(args.dump_outputs, last_loss[0], opt, model, rank)

    # ---- end to end: pinned host batches -> H2D every step, loss -> host every step ----------
    e2e = None
    if not args.no_e2e:
        def endless():
            i = 0
            while True:
                yield wl.host_batches[i % len(wl.host_batches)]
                i += 1
        delay_us = args.upload_delay_us if args.upload_delay_us is not None else (2000.0 if (cuda and step.overlap_update) else 0.0)
        feed = PinnedPrefetcher(endless(), device, upload_delay_us=delay_us)
        loss_host = torch.zeros(args.steps + args.warmup + 4, dtype=torch.float32)
        if cuda:
            loss_host = loss_host.pin_memory()
        k = [0]

        def one():
            loss = step(*wl.to_step_args(next(feed)))
            loss_host[k[0]].copy_(loss.detach().float(), non_blocking=True)   # D2H every step
            k[0] += 1
        for _ in range(min(3, args.warmup)):
            one()
        ms_e2e, _ = timed(one, args.steps)
        sync()
        assert torch.isfinite(loss_host[:k[0]]).all(), "non-finite loss in the end-to-end run"
        ms_e2e = _max_over_ranks(ms_e2e, world)
        e2e = {"value": round(B * world * args.steps / (ms_e2e / 1e3), 2), "unit": wl.unit,
               "h2d_bytes_per_step": int(wl.h2d_bytes), "d2h_bytes_per_step": 4,
               "ms_per_step": round(ms_e2e / args.steps, 4), "upload_delay_us": delay_us}
    clocks = None
    if sampler is not None:
        sampler.stop()
        clocks = sampler.summary(wall0, time.time())      # both timed regions (device-resident and end-to-end) are load

    ms = _max_over_ranks(ms, world)
    value = B * world * args.steps / (ms / 1e3)
    if rank == 0:
        n_params = sum(p.numel() for p in model.parameters())
        cfg = {"model": args.model, "global_batch": B * world, "batch_per_gpu": B, "parallelism": "dp%d" % world,
               "optimizer": "%s lr=%g" % (args.optimizer.upper(), lr), "threshold_mb": args.threshold, "buckets": len(opt.engine.plan.buckets),
               "params": n_params, "backend": dear.backend(), "cuda_graph": bool(step.use_graph),
               "update_overlaps_forward_in_graph": bool(step.overlap_update),
               "l2": "no explicit flush: each step streams activations+weights far larger than the 126 MB L2"}
        if wl.is_bert:
            cfg.update(seq_len=args.sentence_len, fused_dropout_add_ln=wl.fused_ln, tcgen05_ffn=wl.tc_ffn)
        else:
            cfg.update(image=wl.image, channels_last=bool(args.channels_last), fused_bn_relu=getattr(wl, "fused_bn", False))
        out = {
            "metric": wl.metric, "value": round(value, 2), "unit": wl.unit, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None if BASELINE_PUBLISHED is None else round(value / BASELINE_PUBLISHED, 4),
            "dtype": {"fp32": "fp32 (TF32 convolutions, torch defaults, as the reference)", "bf16": "bf16",
                      "amp": "bf16 autocast"}[args.dtype],
            "data": "synthetic", "impl": "dear", "config": cfg, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        }
        print(json.dumps(out), flush=True)
    try:
        step.finish()             # rotated loop: the last update is applied here (outside every timed region)
        opt.engine.close()
    except Exception:             # the measurement is complete and printed: a teardown problem must not void it
        import traceback
        traceback.print_exc()
    dear.shutdown()
    return 0


def _dump_outputs(path, loss, opt, model, rank):
    """--dump-outputs: the loss of the last timed step and the model state after its update."""
    import numpy as np
    import torch
    loss = loss.detach().float().cpu().reshape(1)   # before synchronize(): a replayed graph reuses this buffer
    opt.synchronize()                               # rotated step: applies the update of the last call, on every rank
    if rank != 0:
        return
    state = torch.cat([t.detach().reshape(-1).float() for t in model.state_dict().values() if t.is_floating_point()])
    if state.numel() > DUMP_STATE_SAMPLE:             # one seeded random element from each of DUMP_STATE_SAMPLE equal slices
        edges = torch.arange(DUMP_STATE_SAMPLE + 1, dtype=torch.int64) * state.numel() // DUMP_STATE_SAMPLE
        u = torch.rand(DUMP_STATE_SAMPLE, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
        idx = edges[:-1] + (u * (edges[1:] - edges[:-1])).long()
        state = state[idx.to(state.device)]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "loss.npy"), loss.numpy())
    np.save(os.path.join(path, "model_state.npy"), state.cpu().numpy())


def _max_over_ranks(v, world):
    if world == 1:
        return v
    import torch
    import torch.distributed as dist
    t = torch.tensor([v], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


if __name__ == "__main__":
    sys.exit(main())
